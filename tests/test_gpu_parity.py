"""GPU parity tests: the CUDA path (through the C ABI) against the oracle, the reference-generated golden
vectors, the analytic known answers, and size-independent properties at BASELINE.json's full sizes.

Bar (BASELINE.md §4): |got - want| <= 1e-4 * max|want| on every element whose consistency mask agrees;
elements on the hard threshold may flip and are counted against a budget (tests/util.py)."""
import numpy as np
import pytest
import torch

import magnet_b200
from magnet_b200 import _lib, ops
from magnet_b200.synthetic import make_config, make_inputs
from oracle import magnet_oracle as mo
from tests import kat
from tests.util import compare_volume, golden_inputs, load_golden, oracle_cw

pytestmark = pytest.mark.gpu

VARIANTS = [("direct", _lib.VARIANT_DIRECT), ("cells", _lib.VARIANT_CELLS), ("tma", _lib.VARIANT_TMA),
            ("mma", _lib.VARIANT_MMA)]


def _skip_unsupported(variant, C):
    """The tensor-core kernel is instantiated for C == 64 only (the F-Net width, BASELINE.json configs)."""
    if variant == _lib.VARIANT_MMA and C != 64:
        pytest.skip("MAGNET_VARIANT_MMA: C == 64 only")


def _run_cw(inp, dvol, dev, variant):
    g = inp.to(dev)
    out = magnet_b200.est_costvolume_CW(dvol.to(dev), g.ref_feat, g.nghbr_feat, g.ref_gmms, g.nghbr_gmms, g.R, g.t,
                                        inp.is_valid, inp.cam_intrins, inp.thres, variant=variant)
    torch.cuda.synchronize()
    return out.cpu().numpy()


@pytest.mark.parametrize("vname,variant", VARIANTS)
@pytest.mark.parametrize("name", ["cw_small_random", "cw_small_smooth", "cw_c64_d64", "cw_kitti", "cw_cfg1"])
def test_cw_matches_reference_golden(cuda, name, vname, variant):
    """The reference's own outputs (frozen in tests/golden) are the pin; the oracle supplies flip margins."""
    z, inp = golden_inputs(name)
    _skip_unsupported(variant, inp.ref_feat.shape[1])
    dvol = torch.from_numpy(mo.depth_sampler(inp.ref_gmms[:, 0].numpy(), inp.ref_gmms[:, 1].numpy(), z["k_list"]))
    got = _run_cw(inp, dvol, cuda, variant)
    _, margin = oracle_cw(inp, dvol.numpy(), return_margin=True)
    rep = compare_volume(got, z["cost_cw"], margin, what=f"{name}/{vname}")
    print(name, vname, rep)


@pytest.mark.parametrize("vname,variant", VARIANTS)
@pytest.mark.parametrize("case", sorted(kat.CW_CASES))
def test_cw_known_answers_gpu(cuda, case, vname, variant):
    inp, dvol, exp, tol = kat.CW_CASES[case]()
    _skip_unsupported(variant, inp.ref_feat.shape[1])
    got = _run_cw(inp, dvol, cuda, variant)
    if tol == 0.0:
        assert np.array_equal(got, exp.astype(np.float32))
    else:
        assert np.abs(got - exp).max() <= tol * max(np.abs(exp).max(), 1.0)
    if case == "one_pixel_shift":
        assert np.array_equal(got[..., -1], np.zeros_like(got[..., -1]))


@pytest.mark.parametrize("seed,depth,shape", [
    (21, "random", dict(B=2, V=2, D=5, H=17, W=23, C=16)),       # ragged: HW not a multiple of 32/128
    (22, "smooth", dict(B=1, V=4, D=64, H=30, W=40, C=64)),
    (23, "random", dict(B=1, V=1, D=33, H=9, W=50, C=32)),       # > NCELL cells per lane -> several rounds
    (24, "smooth", dict(B=3, V=3, D=16, H=12, W=12, C=20)),      # C not instantiated by the cells kernel -> direct
    (25, "smooth", dict(B=1, V=2, D=5, H=30, W=40, C=64)),       # the reference's shipped N_s = 5 (one partial chunk)
    (26, "smooth", dict(B=1, V=2, D=80, H=10, W=24, C=32)),      # 2.5 chunks
    (27, "smooth", dict(B=1, V=1, D=256, H=6, W=20, C=16)),      # MAGNET_MAX_PLANES
])
def test_cw_vs_oracle_seeded(cuda, seed, depth, shape):
    inp = make_inputs(seed=seed, depth=depth, invalid=[(0, 0)] if shape["V"] > 1 else (), **shape)
    dvol = inp.depth_volume()
    want, margin = oracle_cw(inp, dvol.numpy(), return_margin=True)
    for vname, variant in VARIANTS:
        if (variant != _lib.VARIANT_DIRECT and shape["C"] not in (16, 32, 64)) or (variant == _lib.VARIANT_MMA and shape["C"] != 64):
            with pytest.raises(_lib.MagnetError):
                _run_cw(inp, dvol, cuda, variant)
            continue
        got = _run_cw(inp, dvol, cuda, variant)
        compare_volume(got, want, margin, what=f"seed{seed}/{vname}")
    got = _run_cw(inp, dvol, cuda, _lib.VARIANT_AUTO)
    compare_volume(got, want, margin, what=f"seed{seed}/auto")


def test_tma_kernel_fuzz_against_direct_kernel(cuda):
    """Randomised shapes / poses for the TMA-staged kernel against the reference-order direct kernel (both depth modes):
    ragged tiles, 1..6 views with invalid ones, 1..150 planes (1..3 chunks, partial lane quarters), large baselines (windows
    that do not fit -> global tap path), random depths (more than 16 cells per pixel -> walk restarts), both families.
    No oracle here, so elements on the consistency threshold are budgeted instead of margin-checked."""
    rng = np.random.default_rng(2024)
    worst = 0.0
    for it in range(24):
        C = int(rng.choice([16, 32, 64]))
        B, V = int(rng.integers(1, 3)), int(rng.integers(1, 7))
        D = int(rng.choice([1, 3, 5, 17, 33, 64, 65, 150])) if it % 3 else int(rng.integers(1, 70))
        H, W = int(rng.integers(5, 41)), int(rng.integers(5, 71))
        depth = "random" if it % 4 == 0 else "smooth"
        family = "kitti" if it % 5 == 0 else "scannet"
        kw = dict(rot_deg=float(rng.uniform(1, 14)), trans=float(rng.uniform(0.05, 0.7))) if it % 2 else {}
        invalid = [(0, int(rng.integers(0, V)))] if V > 1 and it % 3 == 0 else ()
        inp = make_inputs(B=B, V=V, D=D, H=H, W=W, C=C, seed=1000 + it, depth=depth, family=family, invalid=invalid, **kw)
        g = inp.to(cuda)
        plan = magnet_b200.MatchingPlan(g.ref_feat, g.nghbr_feat, g.nghbr_gmms, g.nghbr_poses, inp.is_valid,
                                        inp.cam_intrins, thres=inp.thres)
        k = inp.k.tolist()
        want = plan.cost(g.ref_gmms, k, variant=_lib.VARIANT_DIRECT)
        dvol = ops.sample_depths(g.ref_gmms, k)
        for mode, got in (("fused", plan.cost(g.ref_gmms, k, variant=_lib.VARIANT_TMA)),
                          ("drop-in", magnet_b200.est_costvolume_CW(dvol, g.ref_feat, g.nghbr_feat, g.ref_gmms, g.nghbr_gmms,
                                                                      g.R, g.t, inp.is_valid, inp.cam_intrins, inp.thres,
                                                                      variant=_lib.VARIANT_TMA))):
            assert torch.isfinite(got).all(), (it, mode)
            scale = max(float(want.abs().max()), 1e-20)
            d = (got - want).abs()
            frac = float((d > 1e-4 * scale).float().mean())
            worst = max(worst, frac)
            assert frac <= 2e-3 and float(d.median()) <= 1e-5 * scale, (it, mode, dict(B=B, V=V, D=D, H=H, W=W, C=C, depth=depth), frac)
    print("fuzz: worst fraction of threshold-adjacent elements", worst)


def test_mma_kernel_fuzz_against_direct_kernel(cuda):
    """Randomised shapes / poses for the tensor-core kernel against the reference-order direct kernel (both depth modes):
    ragged tiles, 1..6 views with invalid ones, 1..150 planes (partial and multiple 64-hypothesis chunks), large baselines
    and random depths (windows beyond 256 cells -> sub-windows), both camera families, feature scales from 1e-3 to 1e3
    (the power-of-two split scale).  No oracle here, so elements on the consistency threshold are budgeted."""
    rng = np.random.default_rng(4048)
    worst = 0.0
    for it in range(24):
        B, V = int(rng.integers(1, 3)), int(rng.integers(1, 7))
        D = int(rng.choice([1, 3, 5, 17, 33, 64, 65, 150])) if it % 3 else int(rng.integers(1, 70))
        H, W = int(rng.integers(5, 41)), int(rng.integers(5, 71))
        depth = "random" if it % 4 == 0 else "smooth"
        family = "kitti" if it % 5 == 0 else "scannet"
        kw = dict(rot_deg=float(rng.uniform(1, 14)), trans=float(rng.uniform(0.05, 0.7))) if it % 2 else {}
        invalid = [(0, int(rng.integers(0, V)))] if V > 1 and it % 3 == 0 else ()
        inp = make_inputs(B=B, V=V, D=D, H=H, W=W, C=64, seed=3000 + it, depth=depth, family=family, invalid=invalid, **kw)
        scale = float(10.0 ** rng.integers(-3, 4))
        inp.ref_feat.mul_(scale)
        inp.nghbr_feat.mul_(1.0 / scale if it % 2 else scale)
        g = inp.to(cuda)
        plan = magnet_b200.MatchingPlan(g.ref_feat, g.nghbr_feat, g.nghbr_gmms, g.nghbr_poses, inp.is_valid,
                                        inp.cam_intrins, thres=inp.thres)
        assert plan.layout == _lib.SRC_SPLIT16
        k = inp.k.tolist()
        want = plan.cost(g.ref_gmms, k, variant=_lib.VARIANT_DIRECT)
        dvol = ops.sample_depths(g.ref_gmms, k)
        for mode, got in (("fused", plan.cost(g.ref_gmms, k, variant=_lib.VARIANT_MMA)),
                          ("drop-in", magnet_b200.est_costvolume_CW(dvol, g.ref_feat, g.nghbr_feat, g.ref_gmms, g.nghbr_gmms,
                                                                      g.R, g.t, inp.is_valid, inp.cam_intrins, inp.thres,
                                                                      variant=_lib.VARIANT_MMA))):
            assert torch.isfinite(got).all(), (it, mode)
            sc = max(float(want.abs().max()), 1e-20)
            d = (got - want).abs()
            frac = float((d > 1e-4 * sc).float().mean())
            worst = max(worst, frac)
            assert frac <= 2e-3 and float(d.median()) <= 1e-5 * sc, (it, mode, dict(B=B, V=V, D=D, H=H, W=W, depth=depth), frac)
    print("mma fuzz: worst fraction of threshold-adjacent elements", worst)


def test_mma_launch_is_graph_replayable(cuda):
    """The persistent tensor-core kernel hands out work through a global counter that its last CTA re-arms: a captured
    launch must replay (several times, with new inputs) and agree with an eager launch bit for bit."""
    inp = make_inputs(B=2, V=3, D=64, H=40, W=56, C=64, seed=92, depth="smooth").to(cuda)
    plan = magnet_b200.MatchingPlan(inp.ref_feat, inp.nghbr_feat, inp.nghbr_gmms, inp.nghbr_poses, inp.is_valid,
                                    inp.cam_intrins, thres=5)
    k = ops.k_array(inp.k.tolist())
    gmm = inp.ref_gmms.clone()
    cv = torch.empty(2, 64, 40, 56, device=cuda)
    plan.cost(gmm, k, out=cv)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        plan.cost(gmm, k, out=cv)
    for rep_ in range(3):
        gmm.copy_(inp.ref_gmms * (1.0 + 0.01 * rep_))
        graph.replay()
        torch.cuda.synchronize()
        got = cv.clone()
        want = plan.cost(gmm, k)
        assert torch.equal(got, want), rep_


def test_fused_sampler_equals_drop_in(cuda):
    """MAGNET_DEPTH_GAUSS (sampler fused, analytic cell walk) against MAGNET_DEPTH_VOLUME (drop-in, exact
    per-hypothesis cell walk): d_j is formed with the same separately rounded multiply and add (MAGNET.py:155);
    the two walks may assign a hypothesis that sits on a cell edge to either neighbour, which changes the
    bilinear value by O(1e-6) only (continuity) and can flip an element that sits on the hard threshold."""
    inp = make_inputs(B=2, V=3, D=16, H=24, W=32, C=64, seed=31, depth="smooth")
    g = inp.to(cuda)
    plan = magnet_b200.MatchingPlan(g.ref_feat, g.nghbr_feat, g.nghbr_gmms, g.nghbr_poses, inp.is_valid,
                                    inp.cam_intrins, thres=inp.thres)
    fused = plan.cost(g.ref_gmms, inp.k.tolist())
    dvol = ops.sample_depths(g.ref_gmms, inp.k.tolist())
    assert torch.equal(dvol.cpu(), inp.depth_volume())
    drop = magnet_b200.est_costvolume_CW(dvol, g.ref_feat, g.nghbr_feat, g.ref_gmms, g.nghbr_gmms, g.R, g.t,
                                         inp.is_valid, inp.cam_intrins, inp.thres)
    scale = float(drop.abs().max())
    dd = (fused - drop).abs()
    assert float((dd > 1e-5 * scale).float().mean()) <= 2e-5 and float(dd.median()) <= 1e-6 * scale
    # unsorted offsets disable the analytic walk (exact walk instead): same volume, planes in the other order
    rev = plan.cost(g.ref_gmms, inp.k.tolist()[::-1])
    dr = (rev.flip(1) - fused).abs()
    assert float((dr > 1e-5 * scale).float().mean()) <= 2e-5 and float(dr.median()) <= 1e-6 * scale
    noreuse = plan.cost(g.ref_gmms, inp.k.tolist(), variant=_lib.VARIANT_CELLS_NOREUSE)
    assert torch.equal(plan.cost(g.ref_gmms, inp.k.tolist(), variant=_lib.VARIANT_CELLS), noreuse), \
        "register tap reuse must not change a single bit"
    d_nchw = ops.cost_volume(g.ref_feat, g.nghbr_feat, plan.rays, plan.cams, V=inp.V, src_layout=_lib.SRC_NCHW,
                             consistency=True, src_gmm=g.nghbr_gmms, kappa=5.0, ref_gmm=g.ref_gmms, k=inp.k.tolist(),
                             variant=_lib.VARIANT_DIRECT)
    d_tiled = plan.cost(g.ref_gmms, inp.k.tolist(), variant=_lib.VARIANT_DIRECT)
    assert torch.equal(d_nchw, d_tiled), "TILED32 and NCHW gathers must agree exactly"


@pytest.mark.parametrize("vname,variant", VARIANTS)
@pytest.mark.parametrize("name", ["cw_small_random", "cw_c64_d64", "cw_kitti"])
def test_f_volume_matches_reference_golden(cuda, name, vname, variant):
    z, inp = golden_inputs(name)
    _skip_unsupported(variant, inp.ref_feat.shape[1])
    g = inp.to(cuda)
    dc = torch.from_numpy(z["planes"]).view(1, -1, 1, 1).to(cuda)
    got = magnet_b200.est_costvolume_F(dc, g.ref_feat, g.nghbr_feat, g.R, g.t, inp.is_valid, inp.cam_intrins,
                                       variant=variant).cpu().numpy()
    want = z["cost_f"]
    assert np.abs(got - want).max() <= 1e-4 * np.abs(want).max(), np.abs(got - want).max()
    assert np.allclose(got.sum(axis=1), 1.0, atol=1e-5)


def test_f_identity_uniform_gpu(cuda):
    inp, planes, exp, _ = kat.f_identity()
    g = inp.to(cuda)
    got = magnet_b200.est_costvolume_F(torch.from_numpy(planes).view(1, -1, 1, 1), g.ref_feat, g.nghbr_feat, g.R, g.t,
                                       inp.is_valid, inp.cam_intrins).cpu().numpy()
    assert np.abs(got - exp).max() <= 5e-6      # equal scores up to fp32 rounding -> uniform softmax


def test_update_sampler_kernels_vs_golden(cuda):
    z, _ = load_golden("update_upsample")
    d_out = torch.from_numpy(z["d_output"]).to(cuda).requires_grad_(True)
    ref_gmm = torch.from_numpy(z["ref_gmm"]).to(cuda)
    new = ops.gaussian_update(d_out, ref_gmm)
    (new * torch.from_numpy(z["grad_out"]).to(cuda)).sum().backward()
    assert np.allclose(new.detach().cpu().numpy(), z["new_gmm"], rtol=2e-6, atol=1e-6)
    assert np.allclose(d_out.grad.cpu().numpy(), z["grad_d_output"], rtol=2e-6, atol=1e-6)
    # the GNET mirror is state-dict compatible with the reference's module names and uses the same kernels
    gn = magnet_b200.GNET(ch_in=6).to(cuda)
    assert sorted(gn.state_dict()) == sorted(f"gnet.{i}.{p}" for i in (0, 2, 4, 6) for p in ("weight", "bias"))
    x = torch.randn(2, 6, 9, 11, device=cuda)
    out = gn(x, ref_gmm)
    raw = gn.gnet(x)
    want = mo.gaussian_update(raw.detach().cpu().numpy(), z["ref_gmm"])
    assert np.allclose(out.detach().cpu().numpy(), want, rtol=2e-6, atol=1e-6)
    out.sum().backward()
    assert gn.gnet[6].weight.grad is not None and torch.isfinite(gn.gnet[6].weight.grad).all()


def test_install_rebinds_reference_module(cuda):
    """install() makes a module shaped like models.submodules.homography call the kernels, and the
    reference's loop (restated in oracle/torch_ref.matching_iterations) then runs on them unchanged."""
    import types
    from oracle import torch_ref
    fake = types.ModuleType("models.submodules.homography")
    fake.est_costvolume_CW = torch_ref.cost_volume_cw
    fake.est_costvolume_F = torch_ref.cost_volume_f
    magnet_b200.install(fake)
    assert fake.est_costvolume_CW is magnet_b200.est_costvolume_CW
    inp = make_inputs(B=2, V=2, D=5, H=16, W=24, C=16, seed=41, depth="smooth")
    g = inp.to(cuda)
    torch.manual_seed(0)
    head = magnet_b200.GNET(ch_in=5 + 8).to(cuda)
    x_d3 = torch.randn(2, 8, 16, 24, device=cuda)
    klist = magnet_b200.depth_sampling(3, 5)
    # loop on the B200 kernels (sampler fused, update kernel) ...
    plan = magnet_b200.MatchingPlan(g.ref_feat, g.nghbr_feat, g.nghbr_gmms, g.nghbr_poses, inp.is_valid,
                                    inp.cam_intrins, thres=5)
    ours = magnet_b200.matching_loop(plan, g.ref_gmms, x_d3, head.gnet, 3, klist)
    # ... against the ATen port of the reference loop on the same device (reference-CUDA path)
    theirs = torch_ref.matching_iterations(g, head.gnet, x_d3, 3, klist, 5)
    for a, b in zip(ours[1:], theirs[1:]):
        d = (a - b).abs()
        # a flipped mask element changes one G-Net input; allow a tiny fraction of visibly different pixels
        assert float((d > 1e-3 * b.abs().max()).float().mean()) < 2e-3
        assert float(d.median()) < 1e-5


def test_full_size_properties_cfg2(cuda):
    """BASELINE configs[1] (B=8,V=4,D=64,120x160,C=64): too big for the oracle, so check properties:
    direct and tap-sharing kernels agree; scaling ref features by 2 scales the volume by exactly 2;
    an all-invalid batch element is exactly zero; view order does not matter beyond fp32 summation order."""
    inp = make_config("cfg2", seed=1, invalid=[(3, 0), (3, 1), (3, 2), (3, 3)])
    g = inp.to(cuda)
    plan = magnet_b200.MatchingPlan(g.ref_feat, g.nghbr_feat, g.nghbr_gmms, g.nghbr_poses, inp.is_valid,
                                    inp.cam_intrins, thres=5)
    k = inp.k.tolist()
    cells = plan.cost(g.ref_gmms, k, variant=_lib.VARIANT_TMA)
    direct = plan.cost(g.ref_gmms, k, variant=_lib.VARIANT_DIRECT)
    gather = plan.cost(g.ref_gmms, k, variant=_lib.VARIANT_CELLS)
    assert torch.isfinite(cells).all()
    dg = (gather - direct).abs()
    assert float((dg > 1e-4 * float(direct.abs().max())).float().mean()) <= 3e-5
    assert float(cells[3].abs().max()) == 0.0
    scale = float(direct.abs().max())
    d = (cells - direct).abs()
    frac_bad = float((d > 1e-4 * scale).float().mean())
    print("cfg2 cells-vs-direct: max rel", float(d.max()) / scale, "frac beyond 1e-4", frac_bad,
          "nonzero frac", float((cells != 0).float().mean()))
    assert frac_bad <= 3e-5
    plan2 = magnet_b200.MatchingPlan(g.ref_feat * 2.0, g.nghbr_feat, g.nghbr_gmms, g.nghbr_poses, inp.is_valid,
                                     inp.cam_intrins, thres=5)
    assert torch.equal(plan2.cost(g.ref_gmms, k, variant=_lib.VARIANT_TMA), cells * 2.0)
    # reverse the view order (features, Gaussians, poses, validity all permuted consistently)
    B, V = inp.B, inp.V
    perm = torch.arange(V - 1, -1, -1)
    idx = (perm[:, None] * B + torch.arange(B)[None]).reshape(-1).to(cuda)
    plan3 = magnet_b200.MatchingPlan(g.ref_feat, g.nghbr_feat[idx], g.nghbr_gmms[idx], g.nghbr_poses[:, perm.to(cuda)],
                                     inp.is_valid[:, perm], inp.cam_intrins, thres=5)
    rev = plan3.cost(g.ref_gmms, k, variant=_lib.VARIANT_TMA)
    assert float((rev - cells).abs().max()) <= 2e-6 * scale


@pytest.mark.parametrize("cfg", ["cfg2", "cfg3"])
def test_full_size_vs_reference_operator_sequence(cuda, cfg):
    """What bench.py measures, at BASELINE.json's full sizes (configs[1] and configs[2]): the production kernel in BOTH
    depth modes — sampler fused (MAGNET_DEPTH_GAUSS) and drop-in (d_volume) — against the reference's operator
    sequence (grid_sample / repeat / mul / sum: the ATen port, bit-identical to the reference on the CPU,
    test_oracle_golden.py) on the same device, with consistency-mask flip accounting: an element beyond
    1e-4 * max must sit on the hard threshold (margin from the same operators) and their number is budgeted."""
    from oracle import torch_ref
    from tests.util import FLIP_BUDGET, MARGIN_TOL, REL_TOL
    inp = make_config(cfg, seed=1)
    g = inp.to(cuda)
    cam_d = {k: v.to(cuda) for k, v in inp.cam_intrins.items()}
    with torch.no_grad():
        dvol = ops.sample_depths(g.ref_gmms, inp.k.tolist())
        want = torch_ref.cost_volume_cw(dvol, g.ref_feat, g.nghbr_feat, g.ref_gmms, g.nghbr_gmms, g.R, g.t, inp.is_valid,
                                        cam_d, inp.thres)
        margin = torch_ref.cw_threshold_margin(dvol, g.nghbr_gmms, g.R, g.t, inp.is_valid, cam_d, inp.thres)
        plan = magnet_b200.MatchingPlan(g.ref_feat, g.nghbr_feat, g.nghbr_gmms, g.nghbr_poses, inp.is_valid,
                                        inp.cam_intrins, thres=inp.thres)
        fused = plan.cost(g.ref_gmms, inp.k.tolist())
        drop = magnet_b200.est_costvolume_CW(dvol, g.ref_feat, g.nghbr_feat, g.ref_gmms, g.nghbr_gmms, g.R, g.t,
                                             inp.is_valid, inp.cam_intrins, inp.thres)
    scale = float(want.abs().max())
    for name, got in (("fused", fused), ("drop-in", drop)):
        assert torch.isfinite(got).all()
        diff = (got - want).abs()
        bad = diff > REL_TOL * scale
        n_bad = int(bad.sum())
        far = bad & (margin > MARGIN_TOL)
        print(cfg, name, "max rel on agreeing elements",
              float(torch.where(bad, torch.zeros_like(diff), diff).max()) / scale, "flips", n_bad, "of", got.numel())
        assert not bool(far.any()), f"{cfg}/{name}: {int(far.sum())} elements differ and are NOT on the threshold"
        assert n_bad <= FLIP_BUDGET * got.numel(), f"{cfg}/{name}: flip budget exceeded ({n_bad})"


def test_non_finite_inputs_stated_deviation(cuda):
    """Documented deviation (DESIGN.md "parity"): non-finite source features.  The reference multiplies the sampled
    score by the 0/1 consistency mask, so a NaN / inf feature poisons EVERY hypothesis whose bilinear footprint touches
    it (NaN * 0 = NaN).  The kernels select instead of multiply: a poisoned score that the consistency test rejects
    contributes 0, one that it accepts propagates.  Finite inputs with non-finite POSITIONS (division by ~0) give
    exactly 0 in both.  Pinned here: wherever the reference is finite, the kernel is finite and within the tolerance;
    where the reference is non-finite, the kernel is either non-finite or finite (rejected) — reported, not hidden."""
    from oracle import torch_ref
    for vname, variant in VARIANTS[1:]:
        inp = make_inputs(B=1, V=2, D=16, H=16, W=24, C=64 if variant == _lib.VARIANT_MMA else 16, seed=83, depth="smooth")
        inp.nghbr_feat[0, 3, 5, 7] = float("inf")
        inp.nghbr_feat[1, 0, 9, 11] = float("nan")
        g = inp.to(cuda)
        cam_d = {k: v.to(cuda) for k, v in inp.cam_intrins.items()}
        dvol = inp.depth_volume().to(cuda)
        with torch.no_grad():
            want = torch_ref.cost_volume_cw(dvol, g.ref_feat, g.nghbr_feat, g.ref_gmms, g.nghbr_gmms, g.R, g.t, inp.is_valid,
                                            cam_d, inp.thres)
            got = magnet_b200.est_costvolume_CW(dvol, g.ref_feat, g.nghbr_feat, g.ref_gmms, g.nghbr_gmms, g.R, g.t,
                                                inp.is_valid, inp.cam_intrins, inp.thres, variant=variant)
            fin = torch.isfinite(want)
            assert int((~fin).sum()) > 0, "the case must exercise the non-finite path"
            assert bool(torch.isfinite(got[fin]).all()), f"{vname}: non-finite output where the reference is finite"
            scale = float(want[fin].abs().max())
            d = (got - want).abs()
            assert float((d[fin] > 1e-4 * scale).float().mean()) <= 1e-3, vname
            print(vname, "reference non-finite:", int((~fin).sum()), "of which finite here (rejected by the consistency "
                  "test):", int(torch.isfinite(got[~fin]).sum()))


def test_full_size_identity_known_answer_cfg3(cuda):
    """KITTI-shape grid (B=4,V=4,D=64,88x304): identity pose + open mask => per-pixel dot, every plane."""
    inp = make_config("cfg3", seed=2)
    inp.nghbr_poses.zero_()
    for i in range(4):
        inp.nghbr_poses[:, :, i, i] = 1.0
    inp.nghbr_gmms[:, 1] = 1e6
    g = inp.to(cuda)
    plan = magnet_b200.MatchingPlan(g.ref_feat, g.nghbr_feat, g.nghbr_gmms, g.nghbr_poses, inp.is_valid,
                                    inp.cam_intrins, thres=5)
    got = plan.cost(g.ref_gmms, inp.k.tolist())
    B, V = inp.B, inp.V
    dots = torch.stack([(g.ref_feat * g.nghbr_feat[v * B:(v + 1) * B]).sum(1) for v in range(V)]).mean(0)
    err = (got - dots[:, None]).abs().max()
    assert float(err) <= 1e-4 * float(dots.abs().max())


def test_head_training_step_decreases_loss(cuda):
    """configs[3] in miniature: the head (G-Net + mask head + upsampling) trains through the kernels: gradients
    reach every trainable parameter and a few AdamW steps reduce the Gaussian NLL."""
    import importlib.util, os
    spec = importlib.util.spec_from_file_location("train_head", os.path.join(os.path.dirname(os.path.dirname(__file__)), "examples", "train_head.py"))
    th = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(th)
    inp = make_inputs(B=2, V=2, D=8, H=24, W=32, C=16, seed=51, depth="smooth").to(cuda)
    torch.manual_seed(0)
    head = magnet_b200.MagnetHead(n_samples=8, n_iter=2).to(cuda)
    x_d3 = torch.randn(2, 256, 24, 32, device=cuda)
    gt = torch.nn.functional.interpolate(inp.ref_gmms[:, 0:1] * 1.05, scale_factor=4, mode="nearest")
    opt = torch.optim.AdamW(head.parameters(), lr=1e-3)
    losses = []
    for _ in range(6):
        preds = head(inp.ref_feat, inp.nghbr_feat, inp.ref_gmms, inp.nghbr_gmms, x_d3, inp.nghbr_poses, inp.is_valid, inp.cam_intrins)
        assert len(preds) == 2 and preds[0].shape == (2, 2, 96, 128)
        loss = th.gaussian_nll(preds, gt, gt > 0)
        opt.zero_grad()
        loss.backward()
        assert all(p.grad is not None and torch.isfinite(p.grad).all() for p in head.parameters())
        opt.step()
        losses.append(float(loss))
    assert losses[-1] < losses[0]


@pytest.mark.parametrize("seed,shape,nplanes", [(61, dict(B=2, V=2, D=8, H=20, W=28, C=16), 10),
                                                (62, dict(B=1, V=3, D=12, H=16, W=40, C=64), 10),
                                                # F-Net training shape (train_FNet.py:56-66): 80 SID planes, C=64, 120x160
                                                (63, dict(B=1, V=2, D=8, H=120, W=160, C=64), 80)])
def test_f_volume_backward_matches_autograd_of_reference_ops(cuda, seed, shape, nplanes):
    """SURVEY §8 f-1: gradients of est_costvolume_F w.r.t. both feature maps against autograd through the ATen port
    of the reference (same operator sequence as homography.py:10-75, run on the same device)."""
    from oracle import torch_ref
    inp = make_inputs(seed=seed, depth="smooth", invalid=[(0, 1)], **shape)
    g = inp.to(cuda)
    if nplanes == 80:                                   # SID plane centres as train_FNet.py builds them
        idx = np.arange(81)
        bounds = np.exp(np.log(10.0 + 0.5) * idx / 80) - 0.5
        planes = torch.from_numpy(((bounds[:-1] + bounds[1:]) / 2).astype(np.float32)).to(cuda).view(1, -1, 1, 1)
    else:
        planes = torch.linspace(0.8, 6.0, nplanes, device=cuda).view(1, -1, 1, 1)
    gout = torch.randn(shape["B"], nplanes, shape["H"], shape["W"], device=cuda)
    r1, s1 = g.ref_feat.clone().requires_grad_(True), g.nghbr_feat.clone().requires_grad_(True)
    ours = magnet_b200.est_costvolume_F(planes, r1, s1, g.R, g.t, inp.is_valid, inp.cam_intrins)
    (ours * gout).sum().backward()
    r2, s2 = g.ref_feat.clone().requires_grad_(True), g.nghbr_feat.clone().requires_grad_(True)
    cam_d = {k: v.to(cuda) for k, v in inp.cam_intrins.items()}
    theirs = torch_ref.cost_volume_f(planes, r2, s2, g.R, g.t, inp.is_valid, cam_d)
    (theirs * gout).sum().backward()
    # the outputs are softmax probabilities: a score error d moves a probability by at most d/2, and fp32 re-association
    # of the 64-channel sums is worth ~1e-5 of the largest score (peaked volumes at the F-Net shape: |score| ~ 40)
    with torch.no_grad():
        smax = float(torch_ref.cost_volume_f(planes, g.ref_feat, g.nghbr_feat, g.R, g.t, inp.is_valid, cam_d,
                                             apply_softmax=False).abs().max())
    assert float((ours - theirs).abs().max()) <= max(1e-4 * float(theirs.abs().max()), 1e-5 * smax)
    for a, b, name in ((r1.grad, r2.grad, "ref"), (s1.grad, s2.grad, "src")):
        err = float((a - b).abs().max())
        assert err <= 2e-4 * float(b.abs().max()), (name, err, float(b.abs().max()))


def test_gnet_split_equals_cat_dataflow(cuda):
    """f-3: hoisting the iteration-invariant x_d3 half of G-Net's first convolution out of the loop gives the
    same predictions (and parameter gradients) as the reference's cat([cost, x_d3]) data flow."""
    inp = make_inputs(B=2, V=2, D=8, H=24, W=32, C=16, seed=71, depth="smooth").to(cuda)
    torch.manual_seed(1)
    head = magnet_b200.GNET(ch_in=8 + 256).to(cuda)
    x_d3 = torch.randn(2, 256, 24, 32, device=cuda)
    plan = magnet_b200.MatchingPlan(inp.ref_feat, inp.nghbr_feat, inp.nghbr_gmms, inp.nghbr_poses, inp.is_valid,
                                    inp.cam_intrins, thres=5)
    k = magnet_b200.depth_sampling(3, 8)
    grads = []
    outs = []
    for g_arg in (head.gnet, head):
        head.zero_grad()
        preds = magnet_b200.matching_loop(plan, inp.ref_gmms, x_d3, g_arg, 3, k)
        preds[-1].square().mean().backward()
        outs.append(preds[-1].detach())
        grads.append(torch.cat([p.grad.reshape(-1) for p in head.parameters()]))
    scale = float(outs[0].abs().max())
    d = (outs[0] - outs[1]).abs()
    assert float(d.median()) <= 1e-5 * scale and float((d > 1e-3 * scale).float().mean()) < 2e-3   # mask flips downstream
    assert float((grads[0] - grads[1]).abs().max()) <= 2e-3 * float(grads[0].abs().max())


def test_convex_upsample_kernels_vs_reference(cuda):
    """f-2: fused convex upsampling against the reference's own output (golden) and, for the backward, against
    autograd through the ATen port of upsample_depth_via_mask."""
    from oracle import torch_ref
    z, _ = load_golden("update_upsample")
    depth = torch.from_numpy(z["depth"]).to(cuda).requires_grad_(True)
    mask = torch.from_numpy(z["mask"]).to(cuda).requires_grad_(True)
    up = ops.convex_upsample(depth, mask, 4)
    assert np.allclose(up.detach().cpu().numpy(), z["up"], rtol=1e-5, atol=1e-6)
    g = torch.randn_like(up)
    (up * g).sum().backward()
    d2 = torch.from_numpy(z["depth"]).to(cuda).requires_grad_(True)
    m2 = torch.from_numpy(z["mask"]).to(cuda).requires_grad_(True)
    (torch_ref.convex_upsample(d2, m2, 4) * g).sum().backward()
    assert float((depth.grad - d2.grad).abs().max()) <= 1e-5 * float(d2.grad.abs().max())
    assert float((mask.grad - m2.grad).abs().max()) <= 1e-5 * float(m2.grad.abs().max())


@pytest.mark.parametrize("vname,variant", VARIANTS)
def test_points_behind_the_source_camera(cuda, vname, variant):
    """The reference has no positive-depth test (SURVEY A.5 #3): hypotheses behind a source camera are projected and
    sampled like any other.  A source view translated 3 m forward puts about half of them behind it; the analytic
    cell walk must hand those lanes to the exact walk, and the result must still match the oracle."""
    inp = make_inputs(B=1, V=2, D=32, H=16, W=24, C=64 if variant == _lib.VARIANT_MMA else 16, seed=81, depth="smooth")
    inp.nghbr_poses[0, 0, 2, 3] = -3.0            # z_src = z_ref - 3 < 0 for depths below 3 m
    inp.nghbr_poses[0, 1, 2, 3] = -2.4
    inp.nghbr_gmms[0, 1] = 1e6                    # view 0: consistency test wide open, so behind-camera samples count
    dvol = inp.depth_volume()
    want, margin = oracle_cw(inp, dvol.numpy(), return_margin=True)
    g = inp.to(cuda)
    plan = magnet_b200.MatchingPlan(g.ref_feat, g.nghbr_feat, g.nghbr_gmms, g.nghbr_poses, inp.is_valid,
                                    inp.cam_intrins, thres=5)
    fused = plan.cost(g.ref_gmms, inp.k.tolist(), variant=variant).cpu().numpy()
    compare_volume(fused, want, margin, what=f"behind/{vname}/fused")
    compare_volume(_run_cw(inp, dvol, cuda, variant), want, margin, what=f"behind/{vname}/drop-in")


def test_iteration_is_cuda_graph_capturable(cuda):
    """include/magnet_b200.h promises: no allocation, no synchronisation, every launch on the given stream.  So one
    matching iteration (fused cost kernel + update kernel) must capture into a CUDA graph and replay bit-identically."""
    inp = make_inputs(B=2, V=2, D=16, H=24, W=32, C=32, seed=91, depth="smooth").to(cuda)
    plan = magnet_b200.MatchingPlan(inp.ref_feat, inp.nghbr_feat, inp.nghbr_gmms, inp.nghbr_poses, inp.is_valid,
                                    inp.cam_intrins, thres=5)
    k = ops.k_array(inp.k.tolist())
    raw = torch.randn(2, 2, 24, 32, device=cuda) * 0.1
    cv = torch.empty(2, 16, 24, 32, device=cuda)
    gmm_in = inp.ref_gmms.clone()
    gmm_out = torch.empty_like(gmm_in)

    def iteration():
        plan.cost(gmm_in, k, out=cv)
        gmm_out.copy_(ops.gaussian_update(raw, gmm_in))

    iteration()                                   # warm-up outside capture (one-time function attributes)
    torch.cuda.synchronize()
    eager_cv, eager_gmm = cv.clone(), gmm_out.clone()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(side):
        with torch.cuda.graph(graph, stream=side):
            iteration()
    torch.cuda.current_stream().wait_stream(side)
    cv.zero_()
    gmm_out.zero_()
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(cv, eager_cv) and torch.equal(gmm_out, eager_gmm)
    gmm_in.mul_(1.05)                             # new inputs in the same buffers, replay again
    graph.replay()
    torch.cuda.synchronize()
    want = plan.cost(gmm_in, k)
    assert torch.equal(cv, want)


def test_drop_in_call_is_graph_capturable_and_repacks_inside_the_graph(cuda):
    """VERDICT r1 weak #6: the per-forward preparation cache keys on tensor versions, which a graph replay never bumps.
    While a stream is capturing, est_costvolume_CW therefore bypasses the cache: repack + camera table become graph nodes
    and a replay sees whatever the buffers hold.  (Inputs that live on the CPU cannot be uploaded during capture, so the
    caller passes device-resident cam_intrins / is_valid — the reference's `.item()` on is_valid would not capture at all.)"""
    inp = make_inputs(B=2, V=2, D=16, H=24, W=32, C=32, seed=93, depth="smooth")
    g = inp.to(cuda)
    cam_d = {k: v.to(cuda) for k, v in inp.cam_intrins.items()}
    valid_d = inp.is_valid.to(cuda)
    dvol = inp.depth_volume().to(cuda)
    feat, gmm = g.nghbr_feat.clone(), g.nghbr_gmms.clone()
    out = torch.empty_like(dvol)

    def call():
        out.copy_(magnet_b200.est_costvolume_CW(dvol, g.ref_feat, feat, g.ref_gmms, gmm, g.R, g.t, valid_d, cam_d, inp.thres))

    call()                                                     # warm-up outside capture (function attributes, tensor map path)
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(side):
        with torch.cuda.graph(graph, stream=side):
            call()
    torch.cuda.current_stream().wait_stream(side)
    # refill the source buffers the way a replayed producer would: same tensor objects, new contents
    feat.copy_(g.nghbr_feat.flip(0))
    gmm.copy_(g.nghbr_gmms.flip(0))
    graph.replay()
    torch.cuda.synchronize()
    want = magnet_b200.est_costvolume_CW(dvol, g.ref_feat, g.nghbr_feat.flip(0).contiguous(), g.ref_gmms,
                                         g.nghbr_gmms.flip(0).contiguous(), g.R, g.t, valid_d, cam_d, inp.thres)
    assert torch.equal(out, want), "the replayed graph must repack the refilled buffers, not serve a stale cache entry"


def test_magnet_module_matches_reference_dataflow(cuda):
    """magnet_b200.MAGNET (reference forward signature, backbones injected) against the reference data flow
    (MAGNET.py:130-175) assembled from the ATen port on the same device, with small stand-in backbones."""
    import torch.nn as nn
    from oracle import torch_ref

    class TinyD(nn.Module):                     # (N,3,H,W) -> ((N,2,H/4,W/4) [mu, sigma>0], (N,256,H/4,W/4))
        def __init__(self):
            super().__init__()
            self.a, self.b = nn.Conv2d(3, 2, 4, stride=4), nn.Conv2d(3, 256, 4, stride=4)

        def forward(self, x):
            g = self.a(x)
            return torch.cat([2.5 + 0.5 * torch.tanh(g[:, :1]), 0.2 + 0.05 * torch.sigmoid(g[:, 1:])], 1), self.b(x)

    class TinyF(nn.Module):
        def __init__(self):
            super().__init__()
            self.c = nn.Conv2d(3, 16, 4, stride=4)

        def forward(self, x):
            return self.c(x)

    torch.manual_seed(3)
    B, V, H, W = 2, 2, 96, 128
    inp = make_inputs(B=B, V=V, D=8, H=H // 4, W=W // 4, C=16, seed=95, depth="smooth")
    model = magnet_b200.MAGNET(TinyD(), TinyF(), n_samples=8, weighting="CW5", test_iter=2).to(cuda).eval()
    ref_img = torch.rand(B, 3, H, W, device=cuda)
    nghbr_imgs = torch.rand(V * B, 3, H, W, device=cuda)
    poses = inp.nghbr_poses.to(cuda)
    with torch.no_grad():
        ours = model(ref_img, nghbr_imgs, poses, inp.is_valid, inp.cam_intrins, mode='test')
        # reference data flow on the same tensors
        gm, x_d3 = model.d_net(torch.cat((ref_img, nghbr_imgs), 0))
        feat = model.f_net(torch.cat((ref_img, nghbr_imgs), 0))
        holder = type("H", (), {})()
        holder.ref_feat, holder.nghbr_feat, holder.ref_gmms, holder.nghbr_gmms = feat[:B], feat[B:], gm[:B], gm[B:]
        holder.R, holder.t = poses[:, :, :3, :3], poses[:, :, :3, 3]
        holder.is_valid, holder.cam_intrins = inp.is_valid, {k: v.to(cuda) for k, v in inp.cam_intrins.items()}
        preds = torch_ref.matching_iterations(holder, model.g_net.gnet, x_d3[:B], 2, model.head.k_list, 5)
        mask = model.mask_head(x_d3[:B])
        theirs = [torch_ref.convex_upsample(pr, mask, 4) for pr in preds[1:]]
    assert len(ours) == len(theirs) == 2 and ours[0].shape == (B, 2, H, W)
    for a, b in zip(ours, theirs):
        d = (a - b).abs()
        assert float(d.median()) <= 1e-5 * float(b.abs().max())
        assert float((d > 1e-3 * float(b.abs().max())).float().mean()) < 2e-3     # downstream of rare mask flips


def test_camera_prep_kernels(cuda):
    """f-4: on-device relative poses + validity and grid intrinsics / rays against the REFERENCE's outputs (golden:
    utils.data_preprocess, the ScanNet and the KITTI get_cam_intrinsics); rays / intrinsics bit-identical."""
    from tests.test_oracle_golden import _kitti_raw8
    z, _ = load_golden("camera_prep_loss")
    poses, valid = ops.relative_poses(torch.from_numpy(z["ext_ref"]).to(cuda), torch.from_numpy(z["ext_nghbr"]).to(cuda))
    assert np.array_equal(valid.cpu().numpy(), z["valid"])
    assert np.allclose(poses.cpu().numpy(), z["poses"], rtol=1e-5, atol=2e-6)
    cam = ops.camera_rays(torch.from_numpy(z["scannet_raw"][None]).to(cuda), 120, 160)          # (B,6): ScanNet, no crop
    assert np.array_equal(cam["intM"].cpu().numpy()[0], z["scannet_intM"])
    assert np.array_equal(cam["unit_ray_array_2D"].cpu().numpy()[0], z["scannet_rays"])
    cam = ops.camera_rays(torch.from_numpy(_kitti_raw8(z)).to(cuda), 88, 304)                    # KITTI crop margins
    assert np.array_equal(cam["intM"].cpu().numpy()[0], z["kitti_intM"])
    assert np.array_equal(cam["unit_ray_array_2D"].cpu().numpy()[0], z["kitti_rays"])
    raw = np.array([[1169.6, 1167.1, 646.3, 489.9, 1296.0, 968.0], [577.9, 578.7, 319.5, 239.5, 640.0, 480.0]])
    cam = ops.camera_rays(torch.from_numpy(raw).to(cuda), 120, 160)
    intM, rays = mo.camera_rays(raw, 120, 160)
    assert np.array_equal(cam["intM"].cpu().numpy(), intM)
    assert np.array_equal(cam["unit_ray_array_2D"].cpu().numpy(), rays)


def test_fused_upsample_nll_vs_reference_loss(cuda):
    """f-2: upsampling + gamma-weighted Gaussian NLL fused (no (B,2,4H,4W) tensors) against the loss and the autograd
    gradients the REFERENCE produced (MagnetLoss over upsample_depth_via_mask, golden), including a pixel whose variance
    sits below the 1e-10 clamp."""
    z, _ = load_golden("camera_prep_loss")
    p0 = torch.from_numpy(z["pred0"]).to(cuda).requires_grad_(True)
    p1 = torch.from_numpy(z["pred1"]).to(cuda).requires_grad_(True)
    mask = torch.from_numpy(z["up_mask"]).to(cuda).requires_grad_(True)
    gt, gtm = torch.from_numpy(z["gt"]).to(cuda), torch.from_numpy(z["gt_mask"]).to(cuda)
    loss = ops.magnet_loss([p0, p1], mask, gt, gtm, 4, gamma=0.8)
    loss.backward()
    assert abs(float(loss) - float(z["loss"])) <= 2e-5 * abs(float(z["loss"]))
    for got, want in ((p0.grad, z["g_pred0"]), (p1.grad, z["g_pred1"]), (mask.grad, z["g_mask"])):
        want = torch.from_numpy(want).to(cuda)
        assert float((got - want).abs().max()) <= 2e-5 * float(want.abs().max()), float((got - want).abs().max())
    # and the unfused route of this repo (ConvexUpsample kernels + the NLL in torch) agrees
    import importlib.util, os
    spec = importlib.util.spec_from_file_location("train_head", os.path.join(os.path.dirname(os.path.dirname(__file__)), "examples", "train_head.py"))
    th = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(th)
    ups = [ops.convex_upsample(p.detach(), mask.detach(), 4) for p in (p0, p1)]
    assert abs(float(th.gaussian_nll(ups, gt, gtm)) - float(loss)) <= 2e-5 * abs(float(loss))
