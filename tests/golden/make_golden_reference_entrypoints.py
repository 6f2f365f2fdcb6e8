"""Generates the fixtures that pin the drop-in packages to the original project's own host code
(graphdeco-inria/hierarchical-3d-gaussians; a checkout of it is named by H3DGS_REFERENCE):

  reference_imports.json     every name the reference's Python imports from `diff_gaussian_rasterization` /
                             `gaussian_hierarchy._C`, and the keyword set of each GaussianRasterizationSettings(...) call
                             in gaussian_renderer/__init__.py                (tests/test_reference_imports_cpu.py)
  reference_render.npz       what the reference's render() returns (train_single.py:76-97) and the gradients its autograd
                             graph sends to the parameters, on top of this repo's packages
  reference_render_post.npz  the same for render_post() driven as train_post.py:91-129 drives it
                                                         (both: tests/test_gpu_reference_entrypoints.py)

The kernels run on the emulation build (tests/emul/), on the CPU.  Large outputs are stored as a fixed seeded sample
(SAMPLE_PIXELS pixels, SAMPLE_ROWS parameter rows) with the full array's max |x| as the scale of the comparison.

    H3DGS_REFERENCE=<checkout> python tests/golden/make_golden_reference_entrypoints.py
"""
import json
import os
import re
import sys
import tempfile

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
PKG = os.path.join(ROOT, "hierarchical-3d-gaussians_b200")
for p in (ROOT, PKG, os.path.join(ROOT, "tests"), os.path.join(ROOT, "tests", "emul")):
    sys.path.insert(0, p)

import refharness                                          # noqa: E402
from build_emu import build                                # noqa: E402
from fake_device import cpu_as_device, cuda_names_mean_cpu  # noqa: E402
from h3dgs import synth                                    # noqa: E402
from util import make_scene                                # noqa: E402

SAMPLE_PIXELS = 8192
SAMPLE_ROWS = 1024


def sample(n, k, seed):
    return np.sort(np.random.default_rng(seed).choice(n, min(n, k), replace=False))


def grads_entry(out, params, rows):
    for k, v in params.items():
        g = v.grad.detach().numpy()
        out[f"grad_{k}"] = g[rows]
        out[f"gmax_{k}"] = np.float64(np.abs(g).max())


def reference_render():
    gr = refharness.import_reference_renderer()
    cam, sc, _, _, bg = make_scene(6000, 320, 200, seed=11)
    pc = refharness.StubModel(sc)
    vcam = refharness.StubCamera(cam)
    pkg = gr.render(vcam, pc, refharness.Pipe(), torch.tensor(bg, device="cuda"))
    img, depth = pkg["render"], pkg["depth"]
    g = torch.Generator(device="cpu").manual_seed(0)
    wi = torch.rand(img.shape, generator=g); wd = torch.rand(depth.shape, generator=g)
    ((img * wi).sum() + (depth * wd).sum()).backward()
    pix = sample(cam.H * cam.W, SAMPLE_PIXELS, 0)
    rows = sample(sc["means3D"].shape[0], SAMPLE_ROWS, 1)
    vsp = pkg["viewspace_points"].grad.detach().numpy()
    img, depth = img.detach(), depth.detach()
    out = dict(keys=np.array(sorted(pkg)), pix=pix, rows=rows,
               image=img.numpy().reshape(3, -1)[:, pix], image_max=np.float64(img.abs().max()),
               depth=depth.numpy().reshape(1, -1)[:, pix], depth_max=np.float64(depth.abs().max()),
               n_vis=np.int64(pkg["visibility_filter"].numel()), radii=pkg["radii"].numpy(),
               grad_viewspace_points=vsp[rows], gmax_viewspace_points=np.float64(np.abs(vsp).max()))
    grads_entry(out, pc.params(), rows)
    return out


def reference_render_post():
    from gaussian_hierarchy._C import expand_to_size, get_interpolation_weights
    gr = refharness.import_reference_renderer()
    cam = synth.make_camera(400, 240)
    leaves = synth.cloud_v1(5000, cam, zmin=2.0, zmax=30.0, seed=7, scale_k=1.0)
    z = leaves["means3D"][:, 2:3]
    leaves["scales"] = (5e-3 * np.sqrt(2.0 * z) * np.ones((1, 3))).astype(np.float32)
    h = synth.append_skybox(synth.build_hierarchy(leaves), 200)
    thr = synth.tau_threshold(6.0, cam)
    pc = refharness.StubModel(h)
    vcam = refharness.StubCamera(cam)
    N = pc._xyz.size(0)
    nodes, boxes = torch.tensor(h["nodes"]), torch.tensor(h["boxes"])
    # scratch exactly as train_post.py:59-63
    render_indices = torch.zeros(N).int(); parent_indices = torch.zeros(N).int()
    nodes_for_render_indices = torch.zeros(N).int()
    interpolation_weights = torch.zeros(N).float(); num_siblings = torch.zeros(N).int()
    to_render = expand_to_size(nodes, boxes, thr, vcam.camera_center, torch.zeros((3)), render_indices, parent_indices,
                               nodes_for_render_indices)
    indices = render_indices[:to_render].int()
    get_interpolation_weights(nodes_for_render_indices[:to_render], thr, nodes, boxes, vcam.camera_center.cpu(),
                              torch.zeros((3)), interpolation_weights, num_siblings)
    pkg = gr.render_post(vcam, pc, refharness.Pipe(), torch.zeros(3), render_indices=indices, parent_indices=parent_indices,
                         interpolation_weights=interpolation_weights, num_node_kids=num_siblings, use_trained_exp=True)
    img = pkg["render"]
    g = torch.Generator(device="cpu").manual_seed(1)
    wi = torch.rand(img.shape, generator=g)
    (img * wi).sum().backward()
    pix = sample(cam.H * cam.W, SAMPLE_PIXELS, 0)
    rows = sample(N, SAMPLE_ROWS, 1)
    img = img.detach()
    out = dict(keys=np.array(sorted(pkg)), pix=pix, rows=rows, to_render=np.int64(to_render),
               image=img.numpy().reshape(3, -1)[:, pix], image_max=np.float64(img.abs().max()),
               visibility_filter=pkg["visibility_filter"].numpy())
    grads_entry(out, pc.params(), rows)
    return out


def reference_imports():
    """Every `from <our package> import ...` line of the reference's Python (submodules aside) and the keyword set of
    each GaussianRasterizationSettings(...) call in gaussian_renderer/__init__.py."""
    names = []
    for dp, dns, fns in os.walk(refharness.REF):
        dns[:] = sorted(d for d in dns if d not in ("submodules", ".git"))
        for fn in sorted(fns):
            if fn.endswith(".py"):
                path = os.path.join(dp, fn)
                for m in re.finditer(r"^from ((?:diff_gaussian_rasterization|gaussian_hierarchy)[\w.]*) import (.+)$",
                                     open(path).read(), re.M):
                    for name in m.group(2).split(","):
                        names.append([os.path.relpath(path, refharness.REF), m.group(1), name.strip()])
    text = open(os.path.join(refharness.REF, "gaussian_renderer", "__init__.py")).read()
    calls = re.findall(r"GaussianRasterizationSettings\((.*?)\n    \)", text, re.S)
    return {"imports": names, "settings_keywords": [sorted(re.findall(r"^\s*(\w+)\s*=", c, re.M)) for c in calls]}


def main():
    assert refharness.have_reference(), "set H3DGS_REFERENCE to a checkout of graphdeco-inria/hierarchical-3d-gaussians"
    with open(os.path.join(HERE, "reference_imports.json"), "w") as f:
        json.dump(reference_imports(), f, indent=1)
        f.write("\n")
    with tempfile.TemporaryDirectory() as tmp:
        so = build(tmp)
        with cpu_as_device(so), cuda_names_mean_cpu():
            for name, fn in (("reference_render.npz", reference_render), ("reference_render_post.npz", reference_render_post)):
                np.savez_compressed(os.path.join(HERE, name), **fn())
                print("wrote", name, os.path.getsize(os.path.join(HERE, name)), "bytes")


if __name__ == "__main__":
    main()
