"""GPU: (1) the hierarchy step through the public API (LOD cut -> gather/lerp -> rasterize ->
L1 -> backward) against the oracle composed the same way on the CPU; (2) the tile-shard mode
emulated on one GPU (shards rendered one after the other) equals the unsharded result;
(3) one full-size (1080p) frame: integer artefacts bit-exact, image/gradients within tolerance."""
import numpy as np
import pytest

from h3dgs import synth
from util import rel_err

pytestmark = pytest.mark.gpu


def _oracle_hier_step(h, cam, thr, gt):
    from oracle import oracle
    n, ri, pi, ni = oracle.expand_to_size(h["nodes"], h["boxes"], thr, cam.camera_center)
    ts, kids = oracle.get_interpolation_weights(ni, thr, h["nodes"], h["boxes"], cam.camera_center)
    pi = np.where(pi < 0, ri, pi)
    S = int(h.get("skybox_points", 0))
    if S:                       # skybox rows follow the cut: own parent, t = 1, kids = 1 (render_post :220-234)
        sky = np.arange(h["means3D"].shape[0] - S, h["means3D"].shape[0], dtype=ri.dtype)
        ri, pi = np.concatenate([ri, sky]), np.concatenate([pi, sky])
        ts, kids = np.concatenate([ts, np.ones(S, ts.dtype)]), np.concatenate([kids, np.ones(S, kids.dtype)])
    t = ts[:, None]
    lerp = lambda a: (t.reshape((-1,) + (1,) * (a.ndim - 1)) * a[ri] + (1 - t).reshape((-1,) + (1,) * (a.ndim - 1)) * a[pi]).astype(np.float32)
    qc, qp = h["rotations"][ri], h["rotations"][pi]
    sign = np.where((qc * qp).sum(1, keepdims=True) < 0, -1.0, 1.0).astype(np.float32)
    rots = (t * qc + (1 - t) * qp * sign).astype(np.float32)
    f = oracle.rasterize_forward(lerp(h["means3D"]), lerp(h["shs"]), None, lerp(h["opacities"]), lerp(h["scales"]), rots,
                                 None, cam.world_view_transform, cam.full_proj_transform, cam.camera_center,
                                 np.zeros(3, np.float32), cam.W, cam.H, cam.tanfovx, cam.tanfovy, ts=ts, kids=kids)
    gcol = (np.sign(f["color"] - gt) / gt.size).astype(np.float32)
    b = oracle.rasterize_backward(f, gcol)
    N = h["means3D"].shape[0]
    grads = {}
    for name, key, sgn in [("means3D", "means3D", None), ("scales", "scales", None), ("shs", "sh", None),
                           ("opacities", "opacities", None), ("rotations", "rotations", sign)]:
        g = b[key].astype(np.float64)
        full = np.zeros((N,) + g.shape[1:], np.float64)
        tt = ts.astype(np.float64).reshape((-1,) + (1,) * (g.ndim - 1))
        np.add.at(full, ri, tt * g)
        gp = (1 - tt) * g
        if sgn is not None:
            gp = gp * sgn
        np.add.at(full, pi, gp)
        grads[name] = full
    return n, f, grads


def test_hierarchy_step_matches_oracle_composition():
    import torch
    from h3dgs import pipeline
    cam = synth.make_camera(480, 270)
    leaves = synth.cloud_v1(12000, cam, zmin=2.0, zmax=40.0, seed=3, scale_k=1.0)
    z = leaves["means3D"][:, 2:3]
    leaves["scales"] = (4e-3 * np.sqrt(2.0 * z) * np.exp(0.4 * np.random.default_rng(1).standard_normal((z.shape[0], 3)))).astype(np.float32)
    h = synth.build_hierarchy(leaves)
    thr = synth.tau_threshold(6.0, cam)
    gt = np.random.default_rng(2).uniform(0, 1, (3, cam.H, cam.W)).astype(np.float32)
    n_ref, f, gref = _oracle_hier_step(h, cam, thr, gt)
    assert 0 < n_ref < 12000 * 2 - 1
    scene = pipeline.Scene(h)
    dcam = pipeline.DeviceCamera(cam)
    bg0, gtd = torch.zeros(3, device="cuda"), torch.tensor(gt, device="cuda")
    imgs = {}
    for fused in (False, True):
        # fused=False: the reference's PyTorch gather/lerp around the rasterizer (render_post);
        # fused=True : the same arithmetic inside K1/K9 via settings.render_indices/parent_indices
        loss, radii, n = pipeline.l1_step(scene, dcam, bg0, gtd, thr, fused=fused)
        assert n == n_ref
        assert np.array_equal(radii.cpu().numpy(), f["radii"])
        loss_ref = np.abs(f["color"] - gt).mean()
        assert abs(loss.item() - loss_ref) < 1e-6
        for name, p in [("means3D", scene.means3D), ("scales", scene.scales), ("shs", scene.shs),
                        ("opacities", scene.opacities), ("rotations", scene.rotations)]:
            e = rel_err(p.grad.cpu().numpy(), gref[name])
            assert e < 2e-5, (fused, name, e)          # 1e-5 rasterizer bar + fp32 lerp/scatter
        with torch.no_grad():
            imgs[fused] = (pipeline.render_hier_fused if fused else pipeline.render_hier)(scene, dcam, bg0, thr)[0]
    assert torch.equal(imgs[False], imgs[True])         # bit-identical lerp arithmetic


def test_skybox_rows_follow_the_cut():
    """render_post appends the model's last `skybox_points` rows to every cut with t = 1, kids = 1
    (gaussian_renderer/__init__.py:220-234); both the PyTorch-op form and the fused index form."""
    import torch
    from h3dgs import pipeline
    cam = synth.make_camera(400, 240)
    leaves = synth.cloud_v1(5000, cam, zmin=2.0, zmax=30.0, seed=7, scale_k=1.0)
    z = leaves["means3D"][:, 2:3]
    leaves["scales"] = (5e-3 * np.sqrt(2.0 * z) * np.ones((1, 3))).astype(np.float32)
    h = synth.append_skybox(synth.build_hierarchy(leaves), 300)
    thr = synth.tau_threshold(6.0, cam)
    gt = np.random.default_rng(4).uniform(0, 1, (3, cam.H, cam.W)).astype(np.float32)
    n_ref, f, gref = _oracle_hier_step(h, cam, thr, gt)
    S = h["skybox_points"]
    assert (f["radii"][n_ref:] > 0).sum() > 10            # some of the sky is in view
    scene = pipeline.Scene(h)
    dcam = pipeline.DeviceCamera(cam)
    bg0, gtd = torch.zeros(3, device="cuda"), torch.tensor(gt, device="cuda")
    imgs = {}
    for fused in (False, True):
        loss, radii, n = pipeline.l1_step(scene, dcam, bg0, gtd, thr, fused=fused)
        assert n == n_ref and radii.shape[0] == n + S
        assert np.array_equal(radii.cpu().numpy(), f["radii"])
        assert abs(loss.item() - np.abs(f["color"] - gt).mean()) < 1e-6
        for name, p in [("means3D", scene.means3D), ("scales", scene.scales), ("shs", scene.shs),
                        ("opacities", scene.opacities), ("rotations", scene.rotations)]:
            e = rel_err(p.grad.cpu().numpy(), gref[name])
            assert e < 2e-5, (fused, name, e)
            assert p.grad[-S:].abs().sum() > 0              # the skybox rows receive gradients
        with torch.no_grad():
            imgs[fused] = (pipeline.render_hier_fused if fused else pipeline.render_hier)(scene, dcam, bg0, thr)[0]
    assert torch.equal(imgs[False], imgs[True])


def test_fused_gather_lerp_matches_oracle_directly():
    """op-level: full arrays + render_indices/parent_indices through the public API vs the oracle front-end."""
    import torch
    from oracle import oracle
    from diff_gaussian_rasterization import GaussianRasterizer
    from util import cuda_settings
    cam = synth.make_camera(320, 200)
    leaves = synth.cloud_v1(6000, cam, zmin=2.0, zmax=30.0, seed=2, scale_k=1.0)
    z = leaves["means3D"][:, 2:3]
    leaves["scales"] = (6e-3 * np.sqrt(2 * z) * np.ones((1, 3))).astype(np.float32)
    h = synth.build_hierarchy(leaves)
    thr = synth.tau_threshold(6.0, cam)
    n, ri, pi, ni = oracle.expand_to_size(h["nodes"], h["boxes"], thr, cam.camera_center)
    ts, kids = oracle.get_interpolation_weights(ni, thr, h["nodes"], h["boxes"], cam.camera_center)
    assert (ts < 1).mean() > 0.1
    bg = np.array([0.3, 0.2, 0.1], np.float32)
    f = oracle.rasterize_forward(h["means3D"], h["shs"], None, h["opacities"], h["scales"], h["rotations"], None,
                                 cam.world_view_transform, cam.full_proj_transform, cam.camera_center, bg, cam.W, cam.H,
                                 cam.tanfovx, cam.tanfovy, ts=ts, kids=kids, render_indices=ri, parent_indices=pi)
    gcol = synth.l1_grad(f["color"])
    b = oracle.rasterize_backward(f, gcol)
    rs = cuda_settings(cam, bg, ts=ts, kids=kids)._replace(render_indices=torch.tensor(ri, device="cuda"),
                                                           parent_indices=torch.tensor(pi, device="cuda"))
    t = lambda a: torch.tensor(a, device="cuda", requires_grad=True)
    m, sh, op, s, r = t(h["means3D"]), t(h["shs"]), t(h["opacities"]), t(h["scales"]), t(h["rotations"])
    m2 = torch.zeros((n, 3), device="cuda", requires_grad=True)
    color, radii, _ = GaussianRasterizer(rs)(means3D=m, means2D=m2, shs=sh, colors_precomp=None, opacities=op, scales=s,
                                            rotations=r, cov3D_precomp=None)
    assert np.array_equal(radii.cpu().numpy(), f["radii"])
    assert rel_err(color.detach().cpu().numpy(), f["color"]) < 1e-5
    (color * torch.tensor(gcol, device="cuda")).sum().backward()
    for name, p_ in [("means3D", m), ("sh", sh), ("opacities", op), ("scales", s), ("rotations", r), ("means2D", m2)]:
        e = rel_err(p_.grad.cpu().numpy(), b[name])
        assert e < 1e-5, (name, e)


def test_tile_shards_on_one_gpu_equal_unsharded():
    import torch
    from diff_gaussian_rasterization import _C
    from h3dgs import dist as hd
    from util import make_scene, cuda_settings
    cam, sc, ts, kids, bg = make_scene(5000, 400, 300, mode="hier", seed=9)
    rs = cuda_settings(cam, bg, ts=ts, kids=kids)
    t = lambda a: torch.tensor(a, device="cuda")
    m, sh, op, s, r = t(sc["means3D"]), t(sc["shs"]), t(sc["opacities"]), t(sc["scales"]), t(sc["rotations"])

    def fwd(shard):
        return _C.rasterize_gaussians(rs.bg, m, None, op, s, r, 1.0, None, rs.viewmatrix, rs.projmatrix, rs.tanfovx,
                                      rs.tanfovy, cam.H, cam.W, sh, 3, rs.campos, False, False, None, None,
                                      rs.interpolation_weights, rs.num_node_kids, False, shard=shard)

    def bwd(shard, st, g, phases, scratch=None):
        n, color, radii, gb, bb, ib, _ = st
        return _C.rasterize_gaussians_backward(rs.bg, m, radii, None, op, s, r, 1.0, None, rs.viewmatrix, rs.projmatrix,
                                               rs.tanfovx, rs.tanfovy, g, None, sh, 3, rs.campos, gb, n, bb, ib, False,
                                               None, None, rs.interpolation_weights, rs.num_node_kids, False, cam.H,
                                               cam.W, shard=shard, phases=phases, scratch=scratch)
    full = fwd((1, 0))
    gen = torch.Generator(device=full[1].device).manual_seed(0)
    g = torch.sign(full[1] - torch.rand(full[1].shape, generator=gen, device=full[1].device)) / full[1].numel()
    ref = bwd((1, 0), full, g, 3)
    for world in (2, 3, 8):
        states = [fwd((world, k)) for k in range(world)]
        assert sum(st[0] for st in states) == full[0]                      # every (tile, Gaussian) pair exactly once
        rpr = hd.rows_per_rank(cam.H, world)
        slabs = []
        for k, st in enumerate(states):
            slab = torch.zeros((rpr, 3, 16, cam.W), device="cuda"); slab[:st[1].shape[0]] = st[1]
            slabs.append(slab)
        img = hd.unpack(torch.stack(slabs), cam.H, cam.W, world)
        assert torch.equal(img, full[1])                                   # bit-identical per tile
        P = m.shape[0]
        acc = None
        for k, st in enumerate(states):
            a = bwd((world, k), st, g, 1).view(torch.float32)[: P * 10].clone()
            acc = a if acc is None else acc + a
        scratch = torch.zeros_like(bwd((world, 0), states[0], g, 1))
        scratch.view(torch.float32)[: P * 10] = acc
        out = bwd((world, 0), states[0], g, 2, scratch=scratch)
        for a, b in zip(out, ref):
            if a.numel():
                assert rel_err(a.cpu().numpy(), b.cpu().numpy()) < 1e-5      # only the fp32 sum order differs


def test_full_size_frame_1080p():
    from util import make_scene, oracle_run, cuda_run
    cam, sc, ts, kids, bg = make_scene(300000, 1920, 1080, seed=12, zmax=20.0, scale_k=1.2e-3)
    f, b, gcol, gdep = oracle_run(cam, sc, bg)
    out, g, st = cuda_run(cam, sc, bg, gcol, gdep)
    assert np.array_equal(out["radii"], f["radii"])
    assert np.array_equal(st["keys_sorted"].view(np.uint64), f["keys"])
    assert np.array_equal(st["point_list"].astype(np.uint32), f["point_list"])
    assert np.array_equal(st["ranges"].astype(np.uint32), f["ranges"])
    d = np.abs(out["color"] - f["color"])
    # an alpha that lands within rounding of the 1/255 cut flips a contribution of <= 1/255
    assert (d > 1e-5).mean() < 1e-5 and d.max() < 1.5 / 255
    # 300 k Gaussians, hundreds of blended entries per pixel.  The gradient bar stays 1e-5 per element
    # with the flip allowance of util.assert_grad_close; on top of that the fp32 rounding of the per-pixel
    # quadratic form / exp / T <- T/(1-alpha) recurrence that the published algorithm itself performs
    # leaves up to ~1.6e-5 at this depth against the oracle's exact-arithmetic backward (measured),
    # so this one test states 2e-5.
    from util import assert_grad_close
    for k in ["means3D", "means2D", "sh", "opacities", "scales", "rotations"]:
        assert_grad_close(g[k], b[k], k, tol=2e-5)


def test_config2_size_properties_1M_gaussians_1080p():
    """BASELINE.json configs[1] at full size (1M flat Gaussians, 1920x1080, SH-3), where the CPU oracle is too
    slow to be the checker: size-independent properties of the path instead -- the binned lists are a
    tile-major, depth-sorted partition of exactly sum(tiles_touched) entries; per-pixel state is consistent
    with them; the backward is linear in dL/dcolor."""
    import torch
    from diff_gaussian_rasterization import _C
    cam = synth.make_camera(1920, 1080)
    sc = synth.cloud_v1(1_000_000, cam, sh_degree=3, seed=0)
    t = lambda a: torch.tensor(a, device="cuda")
    m, sh, op, s, r = t(sc["means3D"]), t(sc["shs"]), t(sc["opacities"]), t(sc["scales"]), t(sc["rotations"])
    bg = torch.tensor([0.2, 0.3, 0.4], device="cuda")
    vm, pm, cp = t(cam.world_view_transform), t(cam.full_proj_transform), t(cam.camera_center)
    n, color, radii, gb, bb, ib, _ = _C.rasterize_gaussians(bg, m, None, op, s, r, 1.0, None, vm, pm, cam.tanfovx, cam.tanfovy,
                                                            cam.H, cam.W, sh, 3, cp, False, False)
    sv = _C.state_view(m.shape[0], cam.W, cam.H, n, gb, bb, ib)
    tiles_touched = sv["tiles_touched"].long()
    assert int(tiles_touched.sum()) == n and int(((radii > 0) != (tiles_touched > 0)).sum()) == 0
    keys = sv["keys_sorted"]                                   # int64 view of (tile << 32 | depth bits): all positive
    assert bool((keys[1:] >= keys[:-1]).all())                 # tile-major, depth-sorted
    tile_of = (keys >> 32)
    ranges = sv["ranges"].long()
    T = ranges.shape[0]
    counts = torch.bincount(tile_of, minlength=T)
    assert bool(((ranges[:, 1] - ranges[:, 0]) == counts).all())
    nz = counts > 0
    starts = torch.cumsum(counts, 0) - counts
    assert bool((ranges[nz, 0] == starts[nz]).all()) and int(ranges[:, 1].max()) == n
    pl = sv["point_list"].long()
    assert bool((radii[pl] > 0).all())
    depth_bits = sv["depths"].view(torch.int32).long()
    assert bool(((keys & 0xFFFFFFFF) == depth_bits[pl]).all())
    # per-pixel state
    gx = (cam.W + 15) // 16
    ys, xs = torch.meshgrid(torch.arange(cam.H, device="cuda"), torch.arange(cam.W, device="cuda"), indexing="ij")
    tl = (ys // 16) * gx + xs // 16
    assert bool((sv["n_contrib"].long() <= counts[tl]).all())
    fT = sv["final_T"]
    assert bool(((fT >= 0) & (fT <= 1)).all()) and bool(torch.isfinite(color).all())
    assert bool((color >= 0).all())                            # colours are clamped at 0, bg >= 0
    # linearity of the backward in dL/dcolor
    gen = torch.Generator(device="cuda").manual_seed(0)
    g1 = (torch.rand(color.shape, device="cuda", generator=gen) - 0.5) / color.numel()
    g2 = (torch.rand(color.shape, device="cuda", generator=gen) - 0.5) / color.numel()

    def bwd(g):
        out = _C.rasterize_gaussians_backward(bg, m, radii, None, op, s, r, 1.0, None, vm, pm, cam.tanfovx, cam.tanfovy, g,
                                              None, sh, 3, cp, gb, n, bb, ib, False, None, None, None, None, False,
                                              cam.H, cam.W)
        return [o for o in out if o.numel()]
    a, b, ab = bwd(g1), bwd(g2), bwd(g1 + 2.0 * g2)
    for x, y, z in zip(a, b, ab):
        ref = x + 2.0 * y
        assert float((z - ref).abs().max() / ref.abs().max().clamp_min(1e-30)) < 2e-5
