"""The drop-in against the reference's own forward: magnet_b200.install() rebinds a homography module's operators, and
magnet_b200.MAGNET reproduces what the unmodified MAGNET.forward / GNET.forward / upsample_depth_via_mask computed
(tests/golden/reference_module.npz, made by tests/golden/make_golden.py from the same seeded inputs, weights and
stand-in backbones, fp32 on the CPU)."""
import sys
import types

import pytest
import torch

import magnet_b200
from magnet_b200 import ops
from magnet_b200.synthetic import make_inputs
from oracle import torch_ref
from tests.util import GOLDEN, compare_volume, load_golden, oracle_cw

pytestmark = pytest.mark.gpu

sys.path.insert(0, GOLDEN)
import make_golden as mg  # noqa: E402


def _installed_module():
    """A module object under the reference's name, rebound by install() like the real one."""
    hom = types.ModuleType("models.submodules.homography")
    hom.est_costvolume_CW = hom.est_costvolume_F = None
    magnet_b200.install(hom)
    assert hom.est_costvolume_CW is magnet_b200.est_costvolume_CW
    assert hom.est_costvolume_F is magnet_b200.est_costvolume_F
    return hom


def test_install_and_forward_match_the_reference_golden(cuda, monkeypatch):
    z, _ = load_golden("reference_module")
    inp, ref_img, nghbr_imgs, d_net, f_net = mg.forward_case()
    assert mg.input_digest(inp) == str(z["digest"]), "synthetic generator drifted from the golden fixture"
    B, D = mg.FORWARD_CASE["B"], mg.FORWARD_CASE["D"]
    hom = _installed_module()
    model = magnet_b200.MAGNET(d_net, f_net, n_samples=D, train_iter=mg.FORWARD_ITERS, test_iter=mg.FORWARD_ITERS)
    mg.seed_head(model.g_net, model.mask_head)
    model = model.to(cuda).eval()
    seen = []
    cost = magnet_b200.MatchingPlan.cost

    def spy(self, *a, **k):
        out = cost(self, *a, **k)
        seen.append(out.clone())
        return out

    monkeypatch.setattr(magnet_b200.MatchingPlan, "cost", spy)
    poses = inp.nghbr_poses.to(cuda)
    # the golden side is fp32 on the CPU: keep cuDNN's convolutions in fp32 too (no TF32)
    with torch.no_grad(), torch.backends.cudnn.flags(enabled=True, allow_tf32=False):
        ours = model(ref_img.to(cuda), nghbr_imgs.to(cuda), poses, inp.is_valid, inp.cam_intrins, mode="test")
        feat = model.f_net(torch.cat((ref_img, nghbr_imgs), 0).to(cuda))
    assert len(ours) == mg.FORWARD_ITERS and ours[0].shape == (B, 2, 4 * mg.FORWARD_CASE["H"], 4 * mg.FORWARD_CASE["W"])

    # iteration 0: the reference's depth volume into the drop-in through the installed module; the fused loop's own
    # volume; both agree with the reference's cost volume up to threshold flips (oracle margins)
    dv = ops.sample_depths(inp.ref_gmms.to(cuda), model.head.k_list)
    assert torch.equal(dv.cpu(), torch_ref.sample_depth_candidates(inp.ref_gmms, model.head.k_list))
    g = inp.to(cuda)
    with torch.no_grad():
        cv_drop = hom.est_costvolume_CW(dv, feat[:B], feat[B:], g.ref_gmms, g.nghbr_gmms, g.R, g.t, inp.is_valid,
                                        inp.cam_intrins, 5)
    cv_r = torch.from_numpy(z["cost_cw0"]).to(cuda)
    holder = make_inputs(**mg.FORWARD_CASE)
    holder.ref_feat, holder.nghbr_feat = feat[:B].cpu(), feat[B:].cpu()
    _, margin = oracle_cw(holder, dv.cpu().numpy(), return_margin=True)
    rep = compare_volume(cv_drop.cpu().numpy(), z["cost_cw0"], margin, what="install/iteration0")
    compare_volume(seen[0].cpu().numpy(), z["cost_cw0"], margin, what="fused/iteration0")
    # first prediction (quarter res. Gaussians are upsampled 4x): a pixel may differ visibly only if a flipped
    # cost-volume element lies within the 3x3 receptive field of G-Net's first convolution
    scale = float(cv_r.abs().max())
    flipped = ((seen[0] - cv_r).abs() > 1e-4 * scale).any(1, keepdim=True).float()
    near = torch.nn.functional.max_pool2d(flipped, 3, stride=1, padding=1)
    near_up = torch.nn.functional.interpolate(near, scale_factor=4, mode="nearest") > 0
    near_up = torch.nn.functional.max_pool2d(near_up.float(), 9, stride=1, padding=4) > 0   # + the 3x3 convex upsampling
    idx = mg.forward_sample()
    theirs = torch.from_numpy(z["pred"]).to(cuda)                  # (iterations, sampled pixels, [mu, sigma])
    d0 = (mg.sample_pixels(ours[0], idx) - theirs[0]).abs()
    loud = d0 > 1e-4 * float(z["pred_absmax"][0])
    assert not (loud & ~mg.sample_pixels(near_up.expand(-1, 2, -1, -1), idx)).any(), \
        "a prediction differs where no consistency-mask element flipped"
    for i, pred in enumerate(ours):
        d = (mg.sample_pixels(pred, idx) - theirs[i]).abs()
        top = float(z["pred_absmax"][i])
        assert float(d.median()) <= 1e-5 * top
        assert float((d > 1e-3 * top).float().mean()) < 2e-3
    print("install + forward against the reference:", rep, "loud pixels", int(loud.sum()))


def test_reference_f_volume_through_install(cuda):
    """MAGNET_F.forward's call (MAGNET.py:197-200) through an installed module, forward values against the reference."""
    z, _ = load_golden("reference_module")
    hom = _installed_module()
    inp = make_inputs(**mg.F_CASE)
    assert mg.input_digest(inp) == str(z["f_digest"]), "synthetic generator drifted from the golden fixture"
    g = inp.to(cuda)
    d_center = torch.linspace(*mg.F_CASE_PLANES).view(1, -1, 1, 1).to(cuda)
    with torch.no_grad():
        got = hom.est_costvolume_F(d_center, g.ref_feat, g.nghbr_feat, g.R, g.t, inp.is_valid, inp.cam_intrins)
    want = torch.from_numpy(z["cost_f"]).to(cuda)
    assert float((got - want).abs().max()) <= 1e-4 * float(want.abs().max())
