"""The drop-in tree exposes the reference's import surface (train_tensoIR.py:11-12)."""
import importlib
import os
import sys

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dropin_import_surface():
    sys.path.insert(0, os.path.join(REPO, "dropin"))
    try:
        for m in ("models", "models.tensoRF_rotated_lights", "models.relight_utils", "renderer"):
            sys.modules.pop(m, None)
        rot = importlib.import_module("models.tensoRF_rotated_lights")
        for n in ("raw2alpha", "TensorVMSplit", "AlphaGridMask"):
            assert hasattr(rot, n)
        gen = importlib.import_module("models.tensoRF_general_multi_lights")
        assert issubclass(gen.TensorVMSplit, rot.TensorVMSplit)
        ini = importlib.import_module("models.tensoRF_init")
        assert hasattr(ini, "TensorVMSplit")
        ru = importlib.import_module("models.relight_utils")
        for n in ("render_with_BRDF", "compute_transmittance", "compute_radiance", "GGX_specular",
                  "linear2srgb_torch", "compute_secondary_shading_effects"):
            assert hasattr(ru, n)
        rnd = importlib.import_module("renderer")
        assert hasattr(rnd, "Renderer_TensoIR_train") and hasattr(rnd, "OctreeRender_trilinear_fast")
    finally:
        sys.path.remove(os.path.join(REPO, "dropin"))
        for m in ("models", "models.tensoRF_rotated_lights", "models.tensoRF_general_multi_lights",
                  "models.tensoRF_init", "models.relight_utils", "renderer"):
            sys.modules.pop(m, None)


GOLDEN = os.path.join(REPO, "tests", "golden")


def test_reference_importers_resolve_against_dropin():
    """Every name the reference's own modules import from models.* (dataLoader/tensoIR_rotation_setting.py:13,
    tensoIR_simple.py:12, tensoIR_general_multi_lights.py:13, the train scripts, scripts/relight_importance.py; recorded
    by tests/golden/make_golden.py in reference_imports.json) resolves when dropin/ shadows models/."""
    import json
    with open(os.path.join(GOLDEN, "reference_imports.json")) as fh:
        imports = json.load(fh)
    assert {"dataLoader/tensoIR_rotation_setting.py", "dataLoader/tensoIR_simple.py",
            "dataLoader/tensoIR_general_multi_lights.py", "train_tensoIR.py"} <= set(imports)
    dropin = os.path.join(REPO, "dropin")
    saved = {k: sys.modules.pop(k) for k in list(sys.modules) if k == "models" or k.startswith("models.")}
    sys.path.insert(0, dropin)
    try:
        ru = importlib.import_module("models.relight_utils")
        assert ru.__file__.startswith(dropin)
        for n in ("read_hdr", "Environment_Light", "grid_sample", "compute_visibility",
                  "compute_visibility_and_indirect_light", "sample_ray_equally", "render_with_BRDF", "np", "F", "os"):
            assert hasattr(ru, n), n
        for importer, froms in imports.items():
            for module, names in froms:
                mod = importlib.import_module(module)
                assert mod.__file__.startswith(dropin), (importer, module, mod.__file__)
                for n in names:
                    assert hasattr(mod, n), (importer, module, n)
    finally:
        sys.path.remove(dropin)
        for k in [k for k in sys.modules if k == "models" or k.startswith("models.")]:
            sys.modules.pop(k)
        sys.modules.update(saved)


def test_grid_sample_matches_torch_inside_and_clamps_outside():
    """relight_utils.grid_sample == F.grid_sample(align_corners=True) inside [-1,1]; outside it extrapolates from the
    clamped border taps instead of zero padding (SURVEY.md §8c)."""
    import torch
    import torch.nn.functional as F
    from tensoir_b200.relight_utils import grid_sample
    g = torch.Generator().manual_seed(0)
    img = torch.randn(2, 5, 7, 9, generator=g, requires_grad=True)
    grid = torch.rand(2, 6, 4, 2, generator=g) * 1.96 - 0.98
    a, b = grid_sample(img, grid), F.grid_sample(img, grid, mode="bilinear", padding_mode="zeros", align_corners=True)
    assert torch.allclose(a, b, atol=1e-5)
    ga, = torch.autograd.grad(a.sum(), img)
    gb, = torch.autograd.grad(b.sum(), img)
    assert torch.allclose(ga, gb, atol=1e-5)
    # a W=1 "line": x coordinate beyond the border keeps the border value (weights sum to 1 with clamped taps)
    line = torch.arange(4.).view(1, 1, 4, 1)
    out = grid_sample(line, torch.tensor([[[[0.0, 1.5]]]]))
    assert torch.isfinite(out).all()
    # outside [-1, 1]: the reference's own grid_sample on the same inputs (tests/golden/make_golden.py)
    ref = torch.load(os.path.join(GOLDEN, "grid_sample_outside.pt"), weights_only=True)
    assert float(ref["grid"].abs().max()) > 1.2
    assert torch.allclose(grid_sample(ref["img"], ref["grid"]), ref["out"], atol=1e-5)
