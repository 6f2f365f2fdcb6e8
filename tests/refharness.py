"""TEST INFRASTRUCTURE ONLY.  Runs the reference's OWN, unmodified host code of the path --
`gaussian_renderer.render()` / `render_post()` (gaussian_renderer/__init__.py:20-136, 138-292) --
on top of the drop-in packages of this repo, with a stub `GaussianModel` / camera / pipe that carry exactly the
attributes those two functions read.  Nothing is vendored: the golden-data generators under tests/golden/ put a
checkout of graphdeco-inria/hierarchical-3d-gaussians on sys.path, named by the H3DGS_REFERENCE environment variable;
the tests themselves use only the stubs.

Third-party packages the reference imports that are neither ours nor on this path (simple_knn, plyfile) are stubbed."""
import math
import os
import sys
import types

import numpy as np

REF = os.environ.get("H3DGS_REFERENCE", "")


def have_reference():
    return bool(REF) and os.path.isfile(os.path.join(REF, "gaussian_renderer", "__init__.py"))


def import_reference_renderer():
    """-> the reference's gaussian_renderer module, imported against OUR diff_gaussian_rasterization / gaussian_hierarchy."""
    if "gaussian_renderer" in sys.modules and getattr(sys.modules["gaussian_renderer"], "__file__", "").startswith(REF):
        return sys.modules["gaussian_renderer"]

    def stub(name, **attrs):
        m = types.ModuleType(name)
        for k, v in attrs.items():
            setattr(m, k, v)
        sys.modules.setdefault(name, m)
        return sys.modules[name]
    c = stub("simple_knn._C", distCUDA2=lambda *a, **k: None)
    stub("simple_knn", _C=c)
    stub("plyfile", PlyData=object, PlyElement=object)
    if REF not in sys.path:
        sys.path.append(REF)                   # after the repo's packages: ours shadow nothing of the reference's
    import gaussian_renderer
    assert gaussian_renderer.__file__.startswith(REF), gaussian_renderer.__file__
    import diff_gaussian_rasterization
    assert not diff_gaussian_rasterization.__file__.startswith(REF)
    return gaussian_renderer


class StubModel:
    """The attributes of scene.gaussian_model.GaussianModel that render()/render_post() read
    (get_xyz, get_opacity, get_scaling, get_rotation, get_features, active_sh_degree, max_sh_degree,
    skybox_points, _xyz, pretrained_exposures), holding already-activated values as leaf tensors."""

    def __init__(self, arrays, device="cuda", sh_degree=3, requires_grad=True):
        import torch
        t = lambda a: torch.tensor(np.asarray(a), device=device).requires_grad_(requires_grad)
        self._xyz = t(arrays["means3D"])
        self._scaling = t(arrays["scales"])
        self._rotation = t(arrays["rotations"])
        self._opacity = t(arrays["opacities"])
        self._features = t(arrays["shs"])
        self.active_sh_degree = sh_degree
        self.max_sh_degree = int(round(math.sqrt(arrays["shs"].shape[1]))) - 1
        self.skybox_points = int(arrays.get("skybox_points", 0))
        self.pretrained_exposures = None

    get_xyz = property(lambda s: s._xyz)
    get_scaling = property(lambda s: s._scaling)
    get_rotation = property(lambda s: s._rotation)
    get_opacity = property(lambda s: s._opacity)
    get_features = property(lambda s: s._features)

    def params(self):
        return dict(means3D=self._xyz, scales=self._scaling, rotations=self._rotation, opacities=self._opacity,
                    shs=self._features)


class StubCamera:
    """scene.cameras.Camera as far as the renderers read it (scene/cameras.py:89-98)."""

    def __init__(self, cam, device="cuda"):
        import torch
        self.FoVx = 2.0 * math.atan(cam.tanfovx)
        self.FoVy = 2.0 * math.atan(cam.tanfovy)
        self.image_width, self.image_height = cam.W, cam.H
        self.world_view_transform = torch.tensor(cam.world_view_transform, device=device)
        self.full_proj_transform = torch.tensor(cam.full_proj_transform, device=device)
        self.camera_center = torch.tensor(cam.camera_center, device=device)
        self.image_name = "synthetic"


class Pipe:
    compute_cov3D_python = False
    convert_SHs_python = False
    debug = False
