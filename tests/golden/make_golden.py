"""Generate tests/golden/*.npz by running the UNMODIFIED reference (baegwangbin/MaGNet) on the CPU.

    python tests/golden/make_golden.py <MaGNet checkout> [name ...]

With names, only those files are written (e.g. ``reference_module``); the others stay as committed.

Inputs are not stored: they are rebuilt from the seed by magnet_b200.synthetic (numpy Generator
streams are version-stable); each file carries a sha256 of the inputs so a drifting generator is
detected instead of silently comparing against the wrong reference output.

Reference entry points exercised:
  models/submodules/homography.py  est_costvolume_CW (:79), est_costvolume_F (:10)
  models/MAGNET.py                 GNET.forward update equations (:58-70), upsample_depth_via_mask (:15-27),
                                   MAGNET.depth_sampling (:120-128), the sampler expression (:154-156),
                                   MAGNET.forward (:130-175) with stand-in backbones (reference_module.npz)
"""
import hashlib
import os
import sys
import types

import numpy as np
import torch
import torch.nn as nn

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

CASES = {
    # name: (make_inputs kwargs)
    "cw_small_random": dict(B=2, V=3, D=8, H=24, W=32, C=16, seed=1, depth="random", invalid=[(1, 2)]),
    "cw_small_smooth": dict(B=2, V=3, D=8, H=24, W=32, C=16, seed=2, depth="smooth"),
    "cw_c64_d64": dict(B=1, V=2, D=64, H=16, W=64, C=64, seed=3, depth="smooth"),
    "cw_kitti": dict(B=1, V=2, D=12, H=22, W=76, C=32, seed=4, depth="smooth", family="kitti"),
    "cw_cfg1": dict(B=1, V=2, D=16, H=128, W=160, C=64, seed=0, depth="random"),
}
F_PLANES = 12


def input_digest(inp) -> str:
    h = hashlib.sha256()
    for tsr in (inp.ref_feat, inp.nghbr_feat, inp.ref_gmms, inp.nghbr_gmms, inp.nghbr_poses, inp.is_valid,
                inp.cam_intrins['intM'], inp.cam_intrins['unit_ray_array_2D'], inp.k):
        h.update(np.ascontiguousarray(tsr.numpy()).tobytes())
    return h.hexdigest()


def f_planes(n=F_PLANES, d_min=0.5, d_max=8.0):
    """SID plane centres as train_FNet.py:56-66 builds them (n planes instead of 80)."""
    idx = np.arange(n + 1)
    gamma = 1 - d_min
    bounds = np.exp(np.log(d_max + gamma) * idx / n) - gamma
    return ((bounds[:-1] + bounds[1:]) / 2).astype(np.float32)


# ---- tests/test_gpu_reference_module.py: the reference's MAGNET.forward on stand-in backbones ---------------------
# Quarter-resolution grid of the forward case; images are 4x larger.  Weights and images are drawn from fixed seeds
# (not torch's global RNG), so the reference model here and magnet_b200.MAGNET in the test get identical values.
FORWARD_CASE = dict(B=2, V=3, D=8, H=24, W=32, C=16, seed=97, depth="smooth", invalid=[(1, 2)])
FORWARD_ITERS = 2
FORWARD_SAMPLE = 2048          # full-resolution pixels per prediction kept in the golden file (fixed, seeded)
F_CASE = dict(B=2, V=2, D=8, H=20, W=28, C=16, seed=98, depth="smooth")
F_CASE_PLANES = (0.8, 6.0, 12)  # torch.linspace arguments of d_center
# tests/test_oracle_golden.py: the ATen port against the reference bit for bit (both single-threaded)
PORT_PIN_CASES = ((11, "random"), (12, "smooth"))
PORT_PIN_PLANES = (0.5, 7.0, 9)


def port_pin_inputs(seed, depth):
    from magnet_b200.synthetic import make_inputs
    return make_inputs(B=2, V=2, D=6, H=20, W=28, C=8, seed=seed, depth=depth, invalid=[(0, 1)])


class TinyD(nn.Module):
    """D-Net stand-in: (N,3,H,W) -> (fixed (N,2,H/4,W/4) Gaussians [mu, sigma > 0], (N,256,H/4,W/4) features)."""

    def __init__(self, field):
        super().__init__()
        self.b = nn.Conv2d(3, 256, 4, stride=4)
        self.field = field

    def forward(self, x):
        return self.field.to(x.device), self.b(x)


class TinyF(nn.Module):
    """F-Net stand-in: (N,3,H,W) -> (N,C,H/4,W/4)."""

    def __init__(self, C):
        super().__init__()
        self.c = nn.Conv2d(3, C, 4, stride=4)

    def forward(self, x):
        return self.c(x)


def seed_convs(module, seed):
    """Every Conv2d of ``module`` (in module order) drawn from U(-1/sqrt(fan_in), 1/sqrt(fan_in)) of a seeded generator."""
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for m in module.modules():
            if isinstance(m, nn.Conv2d):
                bound = 1.0 / float(np.sqrt(m.weight[0].numel()))
                m.weight.copy_((torch.rand(m.weight.shape, generator=g) * 2 - 1) * bound)
                m.bias.copy_((torch.rand(m.bias.shape, generator=g) * 2 - 1) * bound)


def forward_case():
    """-> (inputs, ref_img, nghbr_imgs, d_net, f_net) of the forward case, on the CPU."""
    from magnet_b200.synthetic import make_inputs
    inp = make_inputs(**FORWARD_CASE)
    B, V, C = FORWARD_CASE["B"], FORWARD_CASE["V"], FORWARD_CASE["C"]
    H, W = 4 * FORWARD_CASE["H"], 4 * FORWARD_CASE["W"]
    g = torch.Generator().manual_seed(FORWARD_CASE["seed"])
    ref_img = torch.rand(B, 3, H, W, generator=g)
    nghbr_imgs = torch.rand(V * B, 3, H, W, generator=g)
    d_net, f_net = TinyD(torch.cat([inp.ref_gmms, inp.nghbr_gmms], 0)), TinyF(C)
    seed_convs(d_net, 1)
    seed_convs(f_net, 2)
    return inp, ref_img, nghbr_imgs, d_net, f_net


def seed_head(g_net, mask_head):
    seed_convs(g_net, 3)
    seed_convs(mask_head, 4)


def forward_sample():
    """Flat (b, y, x) indices of the full-resolution prediction pixels kept in reference_module.npz."""
    B, H, W = FORWARD_CASE["B"], 4 * FORWARD_CASE["H"], 4 * FORWARD_CASE["W"]
    return np.sort(np.random.default_rng(FORWARD_CASE["seed"]).choice(B * H * W, FORWARD_SAMPLE, replace=False))


def sample_pixels(pred, idx):
    """(B,2,H,W) -> (len(idx), 2) values at flat (b, y, x) indices."""
    B, _, H, W = pred.shape
    return pred.permute(0, 2, 3, 1).reshape(B * H * W, 2)[torch.as_tensor(idx, device=pred.device)]


def import_reference(ref_root):
    if not os.path.isfile(os.path.join(ref_root, "models", "submodules", "homography.py")):
        raise SystemExit(f"{ref_root} is not a MaGNet checkout (no models/submodules/homography.py)")
    sys.path.insert(0, ref_root)
    # utils/utils.py:5-7 imports matplotlib, which is absent; the hot path never touches it.
    for name in ("matplotlib", "matplotlib.pyplot"):
        m = types.ModuleType(name)
        m.use = lambda *a, **k: None
        sys.modules.setdefault(name, m)


def main(ref_root, only=()):
    import_reference(ref_root)
    import models.submodules.homography as refh
    from models.MAGNET import GNET, MAGNET, upsample_depth_via_mask
    from magnet_b200.synthetic import make_inputs

    if only:
        for name in only:
            {"reference_module": reference_module, "torch_port_pin": torch_port_pin}[name]()
        return
    torch.set_num_threads(4)
    for name, kw in CASES.items():
        inp = make_inputs(**kw)
        # the sampler exactly as MAGNET.py:154-156 writes it (k_list = python/numpy floats)
        mu, sigma = torch.split(inp.ref_gmms, 1, dim=1)
        holder = types.SimpleNamespace(sampling_range=3, n_samples=kw["D"])
        k_list = MAGNET.depth_sampling(holder)
        dvol = torch.cat([mu + sigma * k for k in k_list], dim=1)
        out = refh.est_costvolume_CW(dvol, inp.ref_feat, inp.nghbr_feat, inp.ref_gmms, inp.nghbr_gmms,
                                     inp.R, inp.t, inp.is_valid, inp.cam_intrins, inp.thres)
        save = dict(cost_cw=out.numpy(), k_list=np.asarray(k_list, dtype=np.float64),
                    digest=np.array(input_digest(inp)), kwargs=np.array(repr(kw)))
        if name != "cw_cfg1":
            save["d_volume"] = dvol.numpy()
            dc = torch.from_numpy(f_planes()).view(1, F_PLANES, 1, 1)
            save["planes"] = dc.numpy().reshape(-1)
            save["cost_f"] = refh.est_costvolume_F(dc, inp.ref_feat, inp.nghbr_feat, inp.R, inp.t,
                                                    inp.is_valid, inp.cam_intrins).numpy()
        np.savez_compressed(os.path.join(HERE, name + ".npz"), **save)
        print(name, out.shape, "nonzero", float((out != 0).float().mean()))

    # Gaussian update: the reference's GNET.forward with the conv stack replaced by identity,
    # forward value and autograd gradient w.r.t. the (would-be) conv output.
    g = torch.Generator().manual_seed(7)
    d_output = (torch.randn(2, 2, 9, 11, generator=g) * 1.5).requires_grad_(True)
    ref_gmm = torch.stack([torch.rand(2, 9, 11, generator=g) * 4 + 0.5, torch.rand(2, 9, 11, generator=g) + 0.05], 1)
    gn = GNET(ch_in=2)
    gn.gnet = torch.nn.Identity()
    new = gn(d_output, ref_gmm)
    gout = torch.randn(new.shape, generator=g)
    (new * gout).sum().backward()
    # learned convex upsampling
    depth = torch.rand(2, 2, 6, 7, generator=g) * 3
    mask = torch.randn(2, 9 * 16, 6, 7, generator=g)
    up = upsample_depth_via_mask(depth, mask, 4)
    ks = {f"k_{b}_{n}": np.asarray(MAGNET.depth_sampling(types.SimpleNamespace(sampling_range=b, n_samples=n)))
          for (b, n) in ((3, 5), (3, 16), (3, 64), (2, 7))}
    np.savez_compressed(os.path.join(HERE, "update_upsample.npz"),
                        d_output=d_output.detach().numpy(), ref_gmm=ref_gmm.numpy(), new_gmm=new.detach().numpy(),
                        grad_out=gout.numpy(), grad_d_output=d_output.grad.numpy(),
                        depth=depth.numpy(), mask=mask.numpy(), up=up.numpy(), **ks)
    print("update / upsample / k_list written")
    camera_prep_and_loss(g)
    reference_module()
    torch_port_pin()


def reference_module():
    """The reference's MAGNET.forward (MAGNET.py:130-175) in test mode on stand-in backbones, with its iteration-0 cost
    volume, and est_costvolume_F (homography.py:10) through the F-Net call of MAGNET_F.forward (MAGNET.py:197-200)."""
    import models.MAGNET as refm
    import models.submodules.homography as refh
    from magnet_b200.synthetic import make_inputs
    inp, ref_img, nghbr_imgs, d_net, f_net = forward_case()
    M = refm.MAGNET
    m = M.__new__(M)                                 # MAGNET.__init__ without its checkpoint loading (MAGNET.py:73-118)
    nn.Module.__init__(m)
    m.d_net, m.f_net = d_net.eval(), f_net.eval()
    m.sampling_range, m.n_samples, m.weighting = 3, FORWARD_CASE["D"], "CW5"
    m.train_iter = m.test_iter = FORWARD_ITERS
    m.downsample_ratio = 4
    m.k_list = M.depth_sampling(m)
    m.g_net = refm.GNET(ch_in=256 + FORWARD_CASE["D"], ch_out=2)
    h_dim = 128
    m.mask_head = nn.Sequential(nn.Conv2d(256, h_dim, 3, padding=1), nn.ReLU(inplace=True),
                                nn.Conv2d(h_dim, h_dim, 1), nn.ReLU(inplace=True),
                                nn.Conv2d(h_dim, h_dim, 1), nn.ReLU(inplace=True),
                                nn.Conv2d(h_dim, 9 * 4 * 4, 1))
    m.upsample_depth = refm.upsample_depth_via_mask
    seed_head(m.g_net, m.mask_head)
    m.eval()
    seen = []
    cw = refh.est_costvolume_CW

    def spy(*a, **k):
        out = cw(*a, **k)
        seen.append(out.clone())
        return out

    refh.est_costvolume_CW = spy
    try:
        with torch.no_grad():
            preds = m(ref_img, nghbr_imgs, inp.nghbr_poses, inp.is_valid, inp.cam_intrins, mode="test")
    finally:
        refh.est_costvolume_CW = cw
    idx = forward_sample()
    fin = make_inputs(**F_CASE)
    d_center = torch.linspace(*F_CASE_PLANES).view(1, -1, 1, 1)
    with torch.no_grad():
        cost_f = refh.est_costvolume_F(d_center, fin.ref_feat, fin.nghbr_feat, fin.R, fin.t, fin.is_valid,
                                       fin.cam_intrins)
    np.savez_compressed(os.path.join(HERE, "reference_module.npz"),
                        digest=np.array(input_digest(inp)), f_digest=np.array(input_digest(fin)),
                        cost_cw0=seen[0].numpy(), pred=np.stack([sample_pixels(p, idx).numpy() for p in preds]),
                        pred_absmax=np.array([float(p.abs().max()) for p in preds], dtype=np.float32),
                        cost_f=cost_f.numpy())
    print("reference module written:", len(preds), "predictions", tuple(preds[0].shape))


def torch_port_pin():
    """est_costvolume_CW / _F single-threaded: with one thread the ATen kernels give the same bits on AVX2 and
    AVX-512 hosts, so the ATen port can be pinned to these outputs exactly."""
    import models.submodules.homography as refh
    threads = torch.get_num_threads()
    torch.set_num_threads(1)
    save = {}
    try:
        for seed, depth in PORT_PIN_CASES:
            inp = port_pin_inputs(seed, depth)
            dc = torch.linspace(*PORT_PIN_PLANES).view(1, -1, 1, 1)
            save[f"cw_{seed}"] = refh.est_costvolume_CW(inp.depth_volume(), inp.ref_feat, inp.nghbr_feat, inp.ref_gmms,
                                                        inp.nghbr_gmms, inp.R, inp.t, inp.is_valid, inp.cam_intrins,
                                                        5).numpy()
            save[f"f_{seed}"] = refh.est_costvolume_F(dc, inp.ref_feat, inp.nghbr_feat, inp.R, inp.t, inp.is_valid,
                                                      inp.cam_intrins).numpy()
            save[f"digest_{seed}"] = np.array(input_digest(inp))
    finally:
        torch.set_num_threads(threads)
    np.savez_compressed(os.path.join(HERE, "torch_port_pin.npz"), **save)
    print("torch port pin written:", sorted(save))


def _camera_prep_case():
    """(V+1) x B extrinsics with a NaN source pose and a NaN reference pose (same generator as the tests use)."""
    rng = np.random.default_rng(9)
    B, V = 3, 4
    ext = np.tile(np.eye(4, dtype=np.float32), (V + 1, B, 1, 1))
    for f in range(V + 1):
        for b in range(B):
            a = rng.uniform(-0.2, 0.2, 3)
            Rz = np.array([[np.cos(a[0]), -np.sin(a[0]), 0], [np.sin(a[0]), np.cos(a[0]), 0], [0, 0, 1]])
            Ry = np.array([[np.cos(a[1]), 0, np.sin(a[1])], [0, 1, 0], [-np.sin(a[1]), 0, np.cos(a[1])]])
            ext[f, b, :3, :3] = (Rz @ Ry).astype(np.float32)
            ext[f, b, :3, 3] = rng.uniform(-1, 1, 3).astype(np.float32)
    ext_ref, ext_nghbr = ext[V // 2].copy(), np.delete(ext, V // 2, axis=0).copy()
    ext_nghbr[0, 1, 0, 0] = np.nan          # NaN source extrinsic: that view is invalid
    ext_ref[2, 1, 1] = np.nan               # NaN reference extrinsic: all views of that element invalid
    return ext_ref, ext_nghbr


SCANNET_RAW = [1169.621094, 1167.105103, 646.295044, 489.927032, 1296.0, 968.0]      # fx fy cx cy raw_W raw_H
KITTI_RAW = [721.5377, 721.5377, 609.5593, 172.854, 1242.0, 375.0]                    # K_cam2 of a 1242 x 375 drive


def camera_prep_and_loss(g):
    """SURVEY §8 f-4 / f-2 pins: the reference's own data_preprocess (utils/utils.py:72-98), get_cam_intrinsics of the
    ScanNet and KITTI loaders (data/dataloader_scannet.py:113-153, data/dataloader_kitti.py:94-127) and MagnetLoss
    (utils/losses.py:34-50, with autograd gradients through upsample_depth_via_mask)."""
    import tempfile
    import utils.utils as ref_utils
    import utils.losses as ref_losses
    from models.MAGNET import upsample_depth_via_mask
    # numpy 2 cannot take a torch tensor in np.linalg.inv(tensor) the way the 2021 code does (utils.py:92): hand the
    # same values over as an ndarray.  Nothing else of data_preprocess is touched.
    real_inv = np.linalg.inv

    class _NP:
        def __getattr__(self, name):
            return getattr(np, name)

    class _LA:
        def __getattr__(self, name):
            return getattr(np.linalg, name)

        @staticmethod
        def inv(a):
            return real_inv(np.asarray(a))

    shim = _NP()
    shim.linalg = _LA()
    ref_utils.np = shim
    ext_ref, ext_nghbr = _camera_prep_case()
    V, B = ext_nghbr.shape[:2]
    frames = [{"extM": torch.from_numpy(ext_nghbr[v])} for v in range(V)]
    data_array = frames[:V // 2] + [{"extM": torch.from_numpy(ext_ref)}] + frames[V // 2:]
    _, _, poses, valid = ref_utils.data_preprocess(data_array, B)
    ref_utils.np = np

    # ScanNet loader: unbound methods on a stub self, intrinsics from a temp 'intrinsic_color.txt'
    for name in ("pykitti",):
        if name not in sys.modules:
            sys.modules[name] = types.ModuleType(name)
    import data.dataloader_scannet as ds
    import data.dataloader_kitti as dk
    H, W = 120, 160
    stub = types.SimpleNamespace(dpv_H=H, dpv_W=W, raw_WH_dict={"scene0000_00": (int(SCANNET_RAW[4]), int(SCANNET_RAW[5]))})
    cls = ds.ScannetLoadPreprocess
    stub.ray_array = cls.get_ray_array(stub)
    with tempfile.TemporaryDirectory() as td:
        os.makedirs(os.path.join(td, "intrinsic"))
        K4 = np.eye(4)
        K4[0, 0], K4[1, 1], K4[0, 2], K4[1, 2] = SCANNET_RAW[:4]
        with open(os.path.join(td, "intrinsic", "intrinsic_color.txt"), "w") as f:
            for row in K4:
                f.write(" ".join(repr(float(x)) for x in row) + "\n")
        cam_s = cls.get_cam_intrinsics(stub, td, "scene0000_00")
    # KITTI loader: crop to 1216 x 352 (left margin (raw_W-1216)/2, top margin raw_H-352)
    clsk = dk.KittiLoadPreprocess
    Hk, Wk = 88, 304
    stubk = types.SimpleNamespace(dpv_H=Hk, dpv_W=Wk, img_H=352, img_W=1216)
    stubk.ray_array = clsk.get_ray_array(stubk)
    Kk = np.eye(3)
    Kk[0, 0], Kk[1, 1], Kk[0, 2], Kk[1, 2] = KITTI_RAW[:4]
    p_data = types.SimpleNamespace(get_cam2=lambda i: types.SimpleNamespace(size=(int(KITTI_RAW[4]), int(KITTI_RAW[5]))),
                                   calib=types.SimpleNamespace(K_cam2=Kk))
    cam_k = clsk.get_cam_intrinsics(stubk, p_data)

    # MagnetLoss on two upsampled predictions, gradients w.r.t. the quarter-resolution predictions and the mask logits
    preds = [(torch.cat([torch.rand(2, 1, 6, 7, generator=g) * 3 + 0.5, torch.rand(2, 1, 6, 7, generator=g) * 0.4 + 0.05], 1)
              ).requires_grad_(True) for _ in range(2)]
    with torch.no_grad():
        preds[1][0, 1, 2, 3] = 1e-7                       # var below the 1e-10 clamp (losses.py:45)
    mask = torch.randn(2, 9 * 16, 6, 7, generator=g).requires_grad_(True)
    gt = torch.rand(2, 1, 24, 28, generator=g) * 3 + 0.4
    gt_mask = torch.rand(2, 1, 24, 28, generator=g) > 0.3
    loss_fn = ref_losses.MagnetLoss(types.SimpleNamespace(loss_fn="gaussian", loss_gamma=0.8))
    ups = [upsample_depth_via_mask(p, mask, 4) for p in preds]
    loss = loss_fn(ups, gt, gt_mask)
    loss.backward()
    np.savez_compressed(os.path.join(HERE, "camera_prep_loss.npz"),
                        ext_ref=ext_ref, ext_nghbr=ext_nghbr, poses=poses.numpy(), valid=valid.numpy(),
                        scannet_raw=np.asarray(SCANNET_RAW), scannet_intM=cam_s["intM"].numpy(),
                        scannet_rays=cam_s["unit_ray_array_2D"].numpy(),
                        kitti_raw=np.asarray(KITTI_RAW), kitti_intM=cam_k["intM"].numpy(),
                        kitti_rays=cam_k["unit_ray_array_2D"].numpy(),
                        pred0=preds[0].detach().numpy(), pred1=preds[1].detach().numpy(), up_mask=mask.detach().numpy(),
                        gt=gt.numpy(), gt_mask=gt_mask.numpy(), loss=np.float32(loss.item()),
                        g_pred0=preds[0].grad.numpy(), g_pred1=preds[1].grad.numpy(), g_mask=mask.grad.numpy())
    print("camera prep + loss written: valid", valid.tolist(), "loss", float(loss))


if __name__ == "__main__":
    if len(sys.argv) < 2:
        raise SystemExit(__doc__)
    main(sys.argv[1], sys.argv[2:])
