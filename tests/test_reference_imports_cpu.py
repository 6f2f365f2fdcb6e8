"""CPU: every name the original project's Python (graphdeco-inria/hierarchical-3d-gaussians: gaussian_renderer/__init__.py,
scene/gaussian_model.py, train_post.py, render_hierarchy.py) imports from `diff_gaussian_rasterization` and
`gaussian_hierarchy._C` exists in OUR packages, so those modules import against them without modification
(INTEGRATION.md section 1), and each of the three GaussianRasterizationSettings(...) calls in gaussian_renderer/__init__.py
passes exactly our settings fields, all by keyword.  The names and keyword sets were read from the reference's source into
tests/golden/reference_imports.json (tests/golden/make_golden_reference_entrypoints.py)."""
import importlib
import inspect
import json
import os

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "hierarchical-3d-gaussians_b200")


def test_reference_modules_import_against_our_packages(golden_dir):
    with open(os.path.join(golden_dir, "reference_imports.json")) as f:
        ref = json.load(f)
    assert {m for _, m, _ in ref["imports"]} == {"diff_gaussian_rasterization", "gaussian_hierarchy._C"}
    for where, module, name in ref["imports"]:
        obj = getattr(importlib.import_module(module), name, None)
        assert obj is not None, (where, module, name)
        src = inspect.getsourcefile(obj) if inspect.ismodule(obj) else inspect.getsourcefile(inspect.unwrap(obj))
        assert src.startswith(PKG), (where, module, name, src)
    from diff_gaussian_rasterization import GaussianRasterizationSettings
    assert len(ref["settings_keywords"]) == 3, ref["settings_keywords"]
    for kws in ref["settings_keywords"]:
        assert sorted(kws) == sorted(GaussianRasterizationSettings._fields), kws
