"""GPU (or the emulation build: H3DGS_EMULATE=1): the original project's own host code of the path --
`gaussian_renderer.render()` (gaussian_renderer/__init__.py:20-136) and `render_post()` (:138-292), driven as
train_single.py:76-97 / train_post.py:91-129 drive them -- ran unmodified on top of the drop-in packages, and this repo's
own host mirror (GaussianRasterizer, h3dgs.pipeline) produces what it returned from the same seeded inputs.

What the reference returned is stored in tests/golden/reference_render.npz and reference_render_post.npz
(tests/golden/make_golden_reference_entrypoints.py: the same kernels, compiled for the emulator; a fixed seeded sample of
pixels and parameter rows).  Integer outputs compare exactly; images and gradients at the suite's 1e-5 norm-wise bar
(tests/util.py), since fp32 contraction and the atomic sum order differ between the emulator and the device."""
import math

import numpy as np
import pytest

import refharness
from h3dgs import synth
from util import TOL, make_scene

pytestmark = pytest.mark.gpu


def _golden(golden_dir, name):
    z = np.load(f"{golden_dir}/{name}")
    return {k: z[k] for k in z.files}


def _close(ours, ref, scale, what):
    d = np.abs(np.asarray(ours, np.float64) - np.asarray(ref, np.float64)).max()
    assert d <= TOL * max(float(scale), 1e-30), (what, float(d / max(float(scale), 1e-30)))


def _pixels(t, pix):
    a = t.detach().cpu().numpy()
    return a.reshape(a.shape[0], -1)[:, pix]


def test_reference_render_runs_unmodified_on_the_dropin_packages(golden_dir):
    """train_single.py:76,97: render(viewpoint_cam, gaussians, pipe, bg) -> render / depth / viewspace_points /
    visibility_filter / radii; do_depth=True inside."""
    import torch
    from diff_gaussian_rasterization import GaussianRasterizer
    from util import cuda_settings
    ref = _golden(golden_dir, "reference_render.npz")
    assert set(ref["keys"]) == {"render", "depth", "viewspace_points", "visibility_filter", "radii"}
    cam, sc, _, _, bg = make_scene(6000, 320, 200, seed=11)
    vcam = refharness.StubCamera(cam)
    # the reference's call, through this repo's own mirror of the interface
    import types
    cam2 = types.SimpleNamespace(W=cam.W, H=cam.H, world_view_transform=cam.world_view_transform,
                                 full_proj_transform=cam.full_proj_transform, camera_center=cam.camera_center,
                                 tanfovx=math.tan(vcam.FoVx * 0.5), tanfovy=math.tan(vcam.FoVy * 0.5))
    rs = cuda_settings(cam2, bg, 3, do_depth=True)
    pc2 = refharness.StubModel(sc)
    m2d = torch.zeros_like(pc2.get_xyz, requires_grad=True)
    img2, radii2, depth2 = GaussianRasterizer(raster_settings=rs)(
        means3D=pc2.get_xyz, means2D=m2d, shs=pc2.get_features, colors_precomp=None, opacities=pc2.get_opacity,
        scales=pc2.get_scaling, rotations=pc2.get_rotation, cov3D_precomp=None)
    img2 = img2.clamp(0, 1)
    assert img2.shape == (3, cam.H, cam.W) and depth2.shape == (1, cam.H, cam.W)
    _close(_pixels(img2, ref["pix"]), ref["image"], ref["image_max"], "render")
    _close(_pixels(depth2, ref["pix"]), ref["depth"], ref["depth_max"], "depth")
    assert int(ref["n_vis"]) == int((radii2 > 0).sum().item())
    assert np.array_equal(ref["radii"], radii2[radii2 > 0].cpu().numpy())
    g = torch.Generator(device="cpu").manual_seed(0)
    wi = torch.rand(img2.shape, generator=g).to("cuda"); wd = torch.rand(depth2.shape, generator=g).to("cuda")
    ((img2 * wi).sum() + (depth2 * wd).sum()).backward()
    rows = ref["rows"]
    for k, p in pc2.params().items():
        _close(p.grad.cpu().numpy()[rows], ref[f"grad_{k}"], ref[f"gmax_{k}"], k)
    vsp = m2d.grad.cpu().numpy()
    _close(vsp[rows], ref["grad_viewspace_points"], ref["gmax_viewspace_points"], "viewspace_points")
    assert np.abs(ref["grad_means3D"]).max() > 0 and np.abs(vsp[:, :2]).max() > 0 and np.all(vsp[:, 2] == 0)


def test_reference_render_post_runs_unmodified_on_the_dropin_packages(golden_dir):
    """train_post.py:91-129: expand_to_size -> get_interpolation_weights -> render_post(..., render_indices=indices,
    parent_indices, interpolation_weights, num_node_kids) incl. the Python gather / parent lerp / quaternion sign flip /
    skybox rows of :199-234; compared with h3dgs.pipeline.render_hier (PyTorch-op form) and render_hier_fused (K1/K9)."""
    import torch
    from gaussian_hierarchy._C import expand_to_size, get_interpolation_weights
    from h3dgs import pipeline
    ref = _golden(golden_dir, "reference_render_post.npz")
    assert set(ref["keys"]) == {"render", "viewspace_points", "visibility_filter", "radii"}
    cam = synth.make_camera(400, 240)
    leaves = synth.cloud_v1(5000, cam, zmin=2.0, zmax=30.0, seed=7, scale_k=1.0)
    z = leaves["means3D"][:, 2:3]
    leaves["scales"] = (5e-3 * np.sqrt(2.0 * z) * np.ones((1, 3))).astype(np.float32)
    h = synth.append_skybox(synth.build_hierarchy(leaves), 200)
    thr = synth.tau_threshold(6.0, cam)
    vcam = refharness.StubCamera(cam)
    N = h["means3D"].shape[0]
    nodes, boxes = torch.tensor(h["nodes"], device="cuda"), torch.tensor(h["boxes"], device="cuda")
    # the cut the reference's caller computes (train_post.py:59-63, 91-103)
    ri, pi, ni = (torch.zeros(N, dtype=torch.int32, device="cuda") for _ in range(3))
    weights, kids = torch.zeros(N, device="cuda"), torch.zeros(N, dtype=torch.int32, device="cuda")
    to_render = expand_to_size(nodes, boxes, thr, vcam.camera_center, torch.zeros((3)), ri, pi, ni)
    get_interpolation_weights(ni[:to_render], thr, nodes, boxes, vcam.camera_center.cpu(), torch.zeros((3)), weights, kids)
    assert to_render == int(ref["to_render"]) and ref["visibility_filter"].shape[0] == to_render + 200
    assert 0 < to_render < N and float(((weights[:to_render] > 0) & (weights[:to_render] < 1)).float().mean()) > 0.05
    g = torch.Generator(device="cpu").manual_seed(1)
    wi = torch.rand((3, cam.H, cam.W), generator=g).to("cuda")
    bgt = torch.zeros(3, device="cuda")

    scene = pipeline.Scene(h)
    dcam = pipeline.DeviceCamera(cam)
    dcam.tanfovx, dcam.tanfovy = math.tan(vcam.FoVx * 0.5), math.tan(vcam.FoVy * 0.5)
    rows = ref["rows"]
    for fn in (pipeline.render_hier, pipeline.render_hier_fused):
        scene.zero_grad()
        img2, radii2, n2 = fn(scene, dcam, bgt, thr)
        assert n2 == to_render
        img2 = img2.clamp(0, 1)
        _close(_pixels(img2, ref["pix"]), ref["image"], ref["image_max"], (fn.__name__, "render"))
        assert np.array_equal(ref["visibility_filter"], (radii2 > 0).cpu().numpy()), fn.__name__
        (img2 * wi).sum().backward()
        ours = {"means3D": scene.means3D, "scales": scene.scales, "rotations": scene.rotations,
                "opacities": scene.opacities, "shs": scene.shs}
        for k, p in ours.items():
            _close(p.grad.cpu().numpy()[rows], ref[f"grad_{k}"], ref[f"gmax_{k}"], (fn.__name__, k))
