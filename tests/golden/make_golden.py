#!/usr/bin/env python
"""Generate tests/golden/ from the REFERENCE implementation, built into oracle/_ref/ by
oracle/build_ref.py.  The reference is needed only here; the tests read the committed files.

    python tests/golden/make_golden.py            sga_ref_cpu.npz, lga_ref_cpu.npz: input/output vectors
                                                  of the reference's kernel bodies compiled for the host
    python tests/golden/make_golden.py --cpu      ref_cpu_digests.json: the same kernel bodies on the cases
                                                  of tests/test_oracle.py
    python tests/golden/make_golden.py --cuda     ref_cuda_digests.json, ref_cuda_values.npz: the reference
                                                  CUDA extension (needs a GPU) on the cases of
                                                  tests/test_gpu_parity.py, test_gpu_config_shapes.py and
                                                  test_gpu_model_slice.py

The reference ships no golden vectors (SURVEY.md 8c).  Results that the tests compare bit for bit are
kept as SHA-256 digests (tests/util.py digest); results compared within a tolerance as their values at
fixed sample positions plus their largest magnitude (tests/util.py sampled), so that every file stays
small while the inputs -- regenerated from the same seeds by the tests -- can be full size.  A rerun of
--cuda reproduces every digest; the model-slice gradients pass through cuDNN and atomically accumulated
interpolation gradients, so they come out equal to within the test's tolerance, not bit for bit.

    python oracle/build_ref.py --cpu-only && python tests/golden/make_golden.py [--cpu]
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
TESTS = os.path.join(ROOT, "tests")
sys.path.insert(0, ROOT)
sys.path.insert(0, TESTS)
from oracle import ref_cpu  # noqa: E402
from util import case_id, digest, lga_inputs, pack_golden_values, sampled, sga_inputs  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))

SGA_SHAPES = [(2, 3, 7, 5, 6), (1, 2, 1, 4, 3), (1, 1, 2, 1, 5), (1, 2, 3, 6, 1),
              (1, 2, 9, 8, 10), (1, 1, 33, 5, 7)]
LGA_SHAPES = [(2, 7, 5, 6), (1, 3, 9, 11), (1, 1, 1, 1), (1, 2, 3, 5, 4)]


def l1norm(a, axis):
    return (a / np.abs(a).sum(axis=axis, keepdims=True)).astype(np.float32)


def vectors():
    rng = np.random.default_rng(20260923)
    sga = {}
    for k, shape in enumerate(SGA_SHAPES):
        N, C, D, H, W = shape
        x = rng.standard_normal(shape).astype(np.float32)
        g = [l1norm(rng.standard_normal((N, C, 5, H, W)), 2) for _ in range(4)]
        go = rng.standard_normal(shape).astype(np.float32)
        out, mask, temp = ref_cpu.sga_forward(x, *g)
        gi, gg, idx = ref_cpu.sga_backward(x, *g, temp, mask, go)
        sga.update({f"x{k}": x, f"go{k}": go, f"out{k}": out, f"mask{k}": mask.astype(np.uint8),
                    f"left{k}": temp, f"gi{k}": gi, f"idx{k}": idx.astype(np.int32)})
        for d in range(4):
            sga[f"g{k}_{d}"] = g[d]
            sga[f"gg{k}_{d}"] = gg[d]
    np.savez_compressed(os.path.join(HERE, "sga_ref_cpu.npz"), n=len(SGA_SHAPES), **sga)

    lga = {}
    for k, shape in enumerate(LGA_SHAPES):
        x = rng.standard_normal(shape).astype(np.float32)
        fs = shape[:-3] + (75,) + shape[-2:]
        f = l1norm(rng.standard_normal(fs), len(fs) - 3)
        go = rng.standard_normal(shape).astype(np.float32)
        y, y1 = ref_cpu.lga2_forward(x, f, 2)
        gx, gf = ref_cpu.lga2_backward(x, f, y1, go, 2)
        lga.update({f"x{k}": x, f"f{k}": f, f"go{k}": go, f"y{k}": y, f"y1_{k}": y1,
                    f"gx{k}": gx, f"gf{k}": gf})
    np.savez_compressed(os.path.join(HERE, "lga_ref_cpu.npz"), n=len(LGA_SHAPES), **lga)


# ---- the reference's kernel bodies on the host: tests/test_oracle.py ---------------------------------
def _sga_cpu(shape, seed, backward):
    x, g, go = sga_inputs(shape, seed=seed)
    ro, rm, rt = ref_cpu.sga_forward(x, *g)
    d = {"out": digest(ro), "mask": digest(rm, np.uint8), "left": digest(rt)}
    if backward:
        rgi, rgg, ridx = ref_cpu.sga_backward(x, *g, rt, rm, go)
        d.update({"gi": digest(rgi), "idx": digest(ridx, np.int32)})
        d.update({"gg%d" % k: digest(rgg[k]) for k in range(4)})
    return d


def _lga_cpu(shape, seed):
    x, f, go = lga_inputs(shape, seed=seed)
    ry, ry1 = ref_cpu.lga2_forward(x, f)
    rgx, rgf = ref_cpu.lga2_backward(x, f, ry1, go)
    return {"y": digest(ry), "y1": digest(ry1), "gx": digest(rgx), "gf": digest(rgf)}


def cpu_digests(out_dir):
    import test_oracle as T
    rng = np.random.default_rng(20261017)
    # ragged and degenerate volumes, any of D, H, W down to 1; the smallest and largest shape always
    sga_random = [(1, 1, 1, 1, 1), (2, 3, 13, 9, 9)] + \
        [tuple(int(rng.integers(1, hi + 1)) for hi in (2, 3, 13, 9, 9)) for _ in range(28)]
    lga_random = [(1, 1, 1, 1), (2, 7, 8, 8)] + \
        [tuple(int(rng.integers(1, hi + 1)) for hi in (2, 7, 8, 8)) for _ in range(18)]
    out = {
        "sga_kernel_bodies": {case_id(s): _sga_cpu(s, sum(s), np.prod(s) < 200000)
                              for s in T.SGA_BODY_SHAPES},
        "lga_kernel_bodies": {case_id(s): _lga_cpu(s, 3) for s in T.LGA_BODY_SHAPES},
        "sga_random": [],
        "lga_random": [],
    }
    for s in sga_random:
        seed = int(rng.integers(0, 10 ** 6))
        out["sga_random"].append(dict(shape=list(s), seed=seed, **_sga_cpu(s, seed, True)))
    for s in lga_random:
        seed = int(rng.integers(0, 10 ** 6))
        out["lga_random"].append(dict(shape=list(s), seed=seed, **_lga_cpu(s, seed)))
    with open(os.path.join(out_dir, "ref_cpu_digests.json"), "w") as fh:
        json.dump(out, fh, indent=1, sort_keys=True)
        fh.write("\n")


# ---- the reference CUDA extension: the GPU tests ---------------------------------------------------
class _Out:
    def __init__(self):
        self.digests, self.records = {}, {}

    def exact(self, key, t, dtype=np.float32):
        self.digests[key] = digest(t, dtype)

    def close(self, key, t):
        self.records[key] = sampled(t)


def cuda_golden(out_dir):
    import torch
    from oracle import ref_gpu
    import test_gpu_config_shapes as TC
    import test_gpu_model_slice as TM
    import test_gpu_parity as TP

    assert torch.cuda.is_available() and ref_gpu.available()
    o = _Out()

    def cu(a):
        return torch.from_numpy(np.ascontiguousarray(a)).cuda()

    for shape in TP.SGA_SHAPES:
        c = case_id(shape)
        x, g, _ = sga_inputs(shape, seed=1 + sum(shape))
        ro, rm, rt = ref_gpu.sga_forward(cu(x), *[cu(a) for a in g])
        o.exact("sga_forward/%s/out" % c, ro)
        o.exact("sga_forward/%s/mask" % c, rm, np.uint8)
        o.exact("sga_forward/%s/left" % c, rt)
        x, g, go = sga_inputs(shape, seed=3 + sum(shape))
        xt, gt = cu(x), [cu(a) for a in g]
        ro, rm, rt = ref_gpu.sga_forward(xt, *gt)
        rgi, rgg, ridx = ref_gpu.sga_backward(xt, *gt, rt, rm, cu(go))
        o.exact("sga_backward/%s/idx" % c, ridx, np.int32)
        o.close("sga_backward/%s/gi" % c, rgi)
        for d in range(4):
            o.close("sga_backward/%s/gg%d" % (c, d), rgg[d])

    for direction in range(4):
        x, g, _ = sga_inputs(TP.DIRECTION_SHAPE, seed=40 + direction, positive=True)
        g[direction] = (g[direction] * 1.2).astype(np.float32)
        ro, rm, _ = ref_gpu.sga_forward(cu(x), *[cu(a) for a in g])
        assert bool((rm == direction).all())
        o.exact("sga_direction/%d/out" % direction, ro)
        o.exact("sga_direction/%d/mask" % direction, rm, np.uint8)

    for shape in TP.LGA_SHAPES:
        c = case_id(shape)
        x, f, go = lga_inputs(shape, seed=5)
        xt, ft = cu(x), cu(f)
        ry, ry1 = ref_gpu.lga2_forward(xt, ft)
        rgx, rgf = ref_gpu.lga2_backward(xt, ft, ry1, cu(go))
        for k, t in (("y1", ry1), ("y", ry), ("gx", rgx), ("gf", rgf)):
            o.close("lga2/%s/%s" % (c, k), t)

    for fname, passes in TP.LGA_PASSES:
        shape = (1, 2, 6, 9, 12) if "3d" in fname else (2, 6, 9, 12)
        x, f, go = lga_inputs(shape, seed=21 + passes)
        xs = [cu(x)]
        for _ in range(passes):
            xs.append(ref_gpu.lga_forward(xs[-1], cu(f), 2))
        g, gf = cu(go), None
        for k in range(passes - 1, -1, -1):
            g, gf = ref_gpu.lga_backward(xs[k], cu(f), g, gf, 2)
        o.close("lga_passes/%s/y" % fname, xs[-1])
        o.close("lga_passes/%s/gx" % fname, g)
        o.close("lga_passes/%s/gf" % fname, gf)

    a = TP.run_legacy_surface(ref_gpu.module())
    for k, t in zip(("out", "temp", "mask"), a[:3]):
        o.exact("legacy_surface/" + k, t)
    o.exact("legacy_surface/idx", a[5])
    o.close("legacy_surface/gi", a[3])
    for d in range(4):
        o.close("legacy_surface/gg%d" % d, a[4][d])
    o.close("legacy_surface/lga", TP.run_legacy_lga(ref_gpu.module()))

    for name, shape in TC.SGA_CONFIG_SHAPES.items():
        x, g, go = TC.sga_config_inputs(shape)
        ro, rm, rt = ref_gpu.sga_forward(x, *g)
        o.exact("config_sga/%s/out" % name, ro)
        o.exact("config_sga/%s/mask" % name, rm)
        del ro
        rgi, rgg, ridx = ref_gpu.sga_backward(x, *g, rt, rm, go)
        del rt, rm
        o.exact("config_sga/%s/idx" % name, ridx.to(torch.int32), np.int32)
        o.close("config_sga/%s/gi" % name, rgi)
        for k in range(4):
            o.close("config_sga/%s/gg%d" % (name, k), rgg[k])
        del x, g, go, rgi, rgg, ridx
        torch.cuda.empty_cache()

    for name, shape in TC.LGA_CONFIG_SHAPES.items():
        x, f, go = TC.lga_config_inputs(shape)
        ry, ry1 = ref_gpu.lga2_forward(x, f)
        rgx, rgf = ref_gpu.lga2_backward(x, f, ry1, go.clone())
        for k, t in (("y1", ry1), ("y", ry), ("gx", rgx), ("gf", rgf)):
            o.close("config_lga2/%s/%s" % (name, k), t)
        del x, f, go, ry, ry1, rgx, rgf
        torch.cuda.empty_cache()

    for hw in TM.HW:
        c = case_id(hw)
        net, left, right, target = TM.slice_setup(hw)
        ref = TM.SliceNet(use_reference=True).cuda()
        ref.load_state_dict(net.state_dict())
        d, loss, grads = TM.train_step(ref, left, right, target)
        o.close("model_slice/%s/disparity" % c, d)
        o.close("model_slice/%s/loss" % c, np.array([loss], np.float32))
        for k, t in grads.items():
            o.close("model_slice/%s/grad/%s" % (c, k), t)

    torch.cuda.synchronize()
    with open(os.path.join(out_dir, "ref_cuda_digests.json"), "w") as fh:
        json.dump(o.digests, fh, indent=1, sort_keys=True)
        fh.write("\n")
    pack_golden_values(os.path.join(out_dir, "ref_cuda_values.npz"), o.records)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cpu", action="store_true", help="write ref_cpu_digests.json")
    ap.add_argument("--cuda", action="store_true", help="write ref_cuda_digests.json and ref_cuda_values.npz")
    ap.add_argument("--out", default=HERE, help="directory for the --cpu / --cuda files (default: tests/golden)")
    a = ap.parse_args()
    os.makedirs(a.out, exist_ok=True)
    if a.cpu:
        cpu_digests(a.out)
    if a.cuda:
        cuda_golden(a.out)
    if not (a.cpu or a.cuda):
        vectors()
    print("wrote", sorted(os.listdir(a.out if (a.cpu or a.cuda) else HERE)))


if __name__ == "__main__":
    main()
