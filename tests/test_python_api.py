"""Drop-in surface of `diff_gaussian_rasterization` (CPU-checkable parts).

Reference: submodules/diff-gaussian-rasterization-feature/diff_gaussian_rasterization/__init__.py and its
only production caller gaussian_renderer/__init__.py (keyword call sites :75-88,:152-161,:190-203,:243-252).
"""
import ast
import inspect
import json
import os
import re

import pytest
import torch

import diff_gaussian_rasterization as dgr
from diff_gaussian_rasterization import GaussianRasterizationSettings, GaussianRasterizer, rasterize_gaussians

# facts of the reference's sources that the tests below check our surface against; where F3DGS_REFERENCE_ROOT names a
# checkout of the reference project, they are also re-derived from its sources
REF_API = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "reference_api.json")))
REF_ROOT = os.environ.get("F3DGS_REFERENCE_ROOT")


def _settings(**over):
    kw = dict(image_height=32, image_width=32, tanfovx=0.5, tanfovy=0.5, bg=torch.zeros(3), scale_modifier=1.0,
              viewmatrix=torch.eye(4), projmatrix=torch.eye(4), sh_degree=0, campos=torch.zeros(3), prefiltered=False,
              debug=False)
    kw.update(over)
    return GaussianRasterizationSettings(**kw)


def test_public_names():
    for n in ("GaussianRasterizationSettings", "GaussianRasterizer", "rasterize_gaussians", "_RasterizeGaussians",
              "cpu_deep_copy_tuple", "_C"):
        assert hasattr(dgr, n)
    for n in ("rasterize_gaussians", "rasterize_gaussians_backward", "mark_visible"):
        assert hasattr(dgr._C, n)


def test_settings_fields_and_order():
    assert GaussianRasterizationSettings._fields == (
        "image_height", "image_width", "tanfovx", "tanfovy", "bg", "scale_modifier", "viewmatrix", "projmatrix",
        "sh_degree", "campos", "prefiltered", "debug")


def test_forward_signature_matches_reference_keywords():
    params = list(inspect.signature(GaussianRasterizer.forward).parameters)
    assert params == ["self", "means3D", "means2D", "opacities", "shs", "semantic_feature", "colors_precomp",
                      "scales", "rotations", "cov3D_precomp"]
    params = list(inspect.signature(rasterize_gaussians).parameters)
    assert params == ["means3D", "means2D", "sh", "colors_precomp", "semantic_feature", "opacities", "scales",
                      "rotations", "cov3Ds_precomp", "raster_settings"]


def test_argument_validation_raises_like_the_reference():
    r = GaussianRasterizer(_settings())
    P = 4
    m3, m2, op = torch.zeros(P, 3), torch.zeros(P, 3), torch.zeros(P, 1)
    with pytest.raises(Exception, match="SHs or precomputed colors"):
        r(means3D=m3, means2D=m2, opacities=op, scales=torch.ones(P, 3), rotations=torch.ones(P, 4))
    with pytest.raises(Exception, match="SHs or precomputed colors"):
        r(means3D=m3, means2D=m2, opacities=op, shs=torch.zeros(P, 1, 3), colors_precomp=torch.zeros(P, 3),
          scales=torch.ones(P, 3), rotations=torch.ones(P, 4))
    with pytest.raises(Exception, match="scale/rotation pair or precomputed 3D covariance"):
        r(means3D=m3, means2D=m2, opacities=op, shs=torch.zeros(P, 1, 3))
    with pytest.raises(Exception, match="scale/rotation pair or precomputed 3D covariance"):
        r(means3D=m3, means2D=m2, opacities=op, shs=torch.zeros(P, 1, 3), scales=torch.ones(P, 3),
          rotations=torch.ones(P, 4), cov3D_precomp=torch.zeros(P, 6))


def test_no_cpu_fallback_fails_loudly():
    """CPU tensors must raise, never silently run somewhere else."""
    r = GaussianRasterizer(_settings())
    P = 4
    with pytest.raises(RuntimeError, match="CUDA tensor"):
        r(means3D=torch.zeros(P, 3), means2D=torch.zeros(P, 3), opacities=torch.ones(P, 1),
          shs=torch.zeros(P, 1, 3), scales=torch.ones(P, 3), rotations=torch.ones(P, 4),
          semantic_feature=torch.zeros(P, 1, 4))
    with pytest.raises(RuntimeError, match="CUDA tensor"):
        r.markVisible(torch.zeros(P, 3))


def test_bad_means_shape_raises_runtime_error():
    with pytest.raises(RuntimeError, match=r"means3D must have dimensions \(num_points, 3\)"):
        dgr._C.rasterize_gaussians(torch.zeros(3), torch.zeros(5, 2), torch.Tensor([]), torch.Tensor([]),
                                   torch.zeros(5, 1), torch.zeros(5, 3), torch.zeros(5, 4), 1.0, torch.Tensor([]),
                                   torch.eye(4), torch.eye(4), 0.5, 0.5, 8, 8, torch.zeros(5, 1, 3), 0,
                                   torch.zeros(3), False, False)


def test_cpu_deep_copy_tuple():
    t = torch.arange(3.0)
    out = dgr.cpu_deep_copy_tuple((t, 1.5, "x"))
    assert out[1] == 1.5 and out[2] == "x" and torch.equal(out[0], t) and out[0].data_ptr() != t.data_ptr()


def test_every_reference_call_site_binds_to_our_signatures():
    """Bind the keywords of each GaussianRasterizationSettings(...)/rasterizer(...) call of the reference's unmodified
    renderer against our signatures."""
    settings, calls = REF_API["settings_calls"], REF_API["rasterizer_calls"]
    if REF_ROOT:
        tree = ast.parse(open(os.path.join(REF_ROOT, "gaussian_renderer", "__init__.py")).read())
        found = {"GaussianRasterizationSettings": [], "rasterizer": []}
        for node in ast.walk(tree):
            if isinstance(node, ast.Call) and getattr(node.func, "id", None) in found:
                found[node.func.id].append(sorted(k.arg for k in node.keywords))
        assert sorted(found["GaussianRasterizationSettings"]) == sorted(sorted(k) for k in settings)
        assert sorted(found["rasterizer"]) == sorted(sorted(k) for k in calls)
    fwd = inspect.signature(GaussianRasterizer.forward)
    for kws in settings:
        assert set(kws) == set(GaussianRasterizationSettings._fields)
    for kws in calls:
        fwd.bind(None, **{k: None for k in kws})
    assert len(settings) >= 2 and len(calls) >= 2


def test_native_call_arity_matches_reference_wrapper():
    """The reference wrapper calls _C positionally: our binding must take as many arguments as it passes."""
    want = REF_API["wrapper_positional_arities"]
    if REF_ROOT:
        path = os.path.join(REF_ROOT, "submodules", "diff-gaussian-rasterization-feature", "diff_gaussian_rasterization",
                            "__init__.py")
        tree = ast.parse(open(path).read())
        tuples = [n for n in ast.walk(tree) if isinstance(n, ast.Assign) and getattr(n.targets[0], "id", "") == "args"]
        assert sorted(len(t.value.elts) for t in tuples) == sorted(want.values())  # forward, backward
    for name, n in want.items():
        signature = getattr(dgr._C, name).__doc__.strip().splitlines()[0]
        assert len(re.findall(r"\barg\d+:", signature)) == n, (name, signature)
