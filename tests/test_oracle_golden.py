"""The oracle restatement vs. outputs of the real reference (fixtures made by
tests/golden/make_golden.py).  CPU only; bit-exact unless stated."""
import torch

from oracle import tensoir_oracle as O
from helpers import oracle_field, named_oracle_params


def eq(a, b, tol=0.0):
    if a is None or b is None:
        assert a is None and b is None
        return
    if a.dtype == torch.bool:
        assert torch.equal(a, b)
        return
    if tol == 0.0:
        assert torch.equal(a, b), float((a - b).abs().max())
    else:
        assert torch.allclose(a, b, rtol=tol, atol=tol), float((a - b).abs().max())


def test_unit_functions(golden_rotated):
    fx = golden_rotated
    f = oracle_field(fx)
    pts = fx["pts"]
    xn = O.normalize_coord(f, pts)
    eq(O.sample_alpha(f, pts), fx["sample_alpha"])
    eq(O.density_feature(f, xn), fx["density_feature"])
    eq(O.feature2density(f, O.density_feature(f, xn)), fx["sigma"])
    rad, intr = O.both_feature(f, xn, fx["li"])
    eq(rad, fx["rad_feat"])
    eq(intr, fx["intr_feat"])
    eq(O.app_feature(f, xn, fx["li"]), fx["app_feat"])
    eq(O.intrin_feature(f, xn), fx["intrin_only"])
    eq(O.mlp_render_fea(f, f.mlp_rgb, fx["viewdirs"], rad), fx["mlp_rgb"])
    eq(O.mlp_pe_and_feature(f, f.mlp_brdf, xn, intr, torch.sigmoid), fx["mlp_brdf"])
    eq(O.mlp_pe_and_feature(f, f.mlp_normal, xn, intr, torch.tanh), fx["mlp_normal"])
    eq(O.derived_normals(f, fx["xj"].clone()).detach(), fx["derived_normals"])


def test_sample_ray(golden_rotated):
    fx = golden_rotated
    f = oracle_field(fx)
    rays = fx["rays"]
    assert f.derived()[4] == fx["nSamples"]
    for got, want in zip(O.sample_ray(f, rays[:, :3], rays[:, 3:6], False, -1), fx["sample_ray_eval"]):
        eq(got, want)
    for got, want in zip(O.sample_ray(f, rays[:, :3], rays[:, 3:6], True, 40, jitter=fx["jitter40"]),
                         fx["sample_ray_train"]):
        eq(got, want)


def test_secondary(golden_rotated):
    fx = golden_rotated
    f = oracle_field(fx)
    got = O.compute_transmittance(f, fx["surf"], fx["dirs"], 96, 0.05, 1.5)
    for g, w in zip(got, fx["transmittance"]):
        eq(g, w)
    got = O.compute_radiance(f, fx["surf"], fx["dirs"], fx["li2"], 96, 0.05, 1.5)
    for g, w in zip(got, fx["radiance"]):
        eq(g, w)
    assert f.counters["density"] > 0 and f.counters["app"] > 0


def test_primary_eval(golden_rotated):
    fx = golden_rotated
    f = oracle_field(fx)
    torch.manual_seed(101)
    got = O.primary_forward(f, fx["rays"], fx["light_idx"], True, False, True, -1)
    for g, w in zip(got, fx["primary_eval"]):
        eq(g.detach() if torch.is_tensor(g) else g, w)
    got = O.primary_forward(f, fx["rays"], fx["light_idx"], True, False, False, -1)
    for g, w in zip(got, fx["primary_eval_norelight"]):
        eq(g.detach() if torch.is_tensor(g) else g, w)


def test_lights_and_brdf(golden_rotated):
    fx = golden_rotated
    f = oracle_field(fx)
    eq(O.gen_light_incident_dirs(f, 'fixed_envirmap'), fx["fixed_dirs"])
    eq(O.generate_envir_map_dir(16, 32)[0], fx["area_weight"])
    eq(O.get_light_rgbs(f, fx["fixed_dirs"]).detach(), fx["light_rgbs"])
    nrm, v2c, rough, fres = fx["ggx_in"]
    eq(O.ggx_specular(nrm, v2c, fx["fixed_dirs"][None].repeat(9, 1, 1), rough, fres), fx["ggx"])


def test_boundary_eval(golden_rotated):
    fx = golden_rotated
    f = oracle_field(fx)
    torch.manual_seed(102)
    got = O.renderer_train(f, fx["rays"], fx["light_idx"], -1, True, False, True, 'fixed_envirmap', 160000, 24)
    for k, w in fx["renderer_eval"].items():
        eq(got[k].detach(), w)


def test_boundary_train_with_grads(golden_rotated):
    """Same seed => same random stream (jitter, xyz noise, light jitter drawn in reference order)."""
    fx = golden_rotated
    f = oracle_field(fx, requires_grad=True)
    torch.manual_seed(fx["train_seed"])
    got = O.renderer_train(f, fx["rays"], fx["light_idx"], 60, True, True, True, 'stratified_sampling', 160000, 24)
    for k, w in fx["renderer_train"].items():
        eq(got[k].detach(), w)
    target = torch.full_like(got["rgb_map"], 0.5)
    loss = (((got["rgb_map"] - target) ** 2).mean() + 0.2 * ((got["rgb_with_brdf_map"] - target) ** 2).mean()
            + 0.0005 * got["normals_diff_map"].mean() + 0.001 * got["normals_orientation_loss_map"].mean()
            + 0.001 * got["albedo_smoothness_loss"] + 0.001 * got["roughness_smoothness_loss"])
    loss.backward()
    eq(loss.detach(), fx["renderer_train_loss"])
    params = named_oracle_params(f)
    n_checked = 0
    for k, g in fx["renderer_train_grads_sample"].items():
        if g is None:
            assert params[k].grad is None or float(params[k].grad.abs().max()) == 0.0
            continue
        eq(params[k].grad.reshape(-1)[g["idx"].long()], g["val"], tol=1e-6)
        eq(params[k].grad.abs().max(), g["absmax"], tol=1e-6)
        n_checked += 1
    assert n_checked >= 20


def test_general_model_boundary(golden_general):
    fx = golden_general
    f = oracle_field(fx)
    torch.manual_seed(103)
    got = O.renderer_train(f, fx["rays"], fx["light_idx"], -1, True, False, True, 'fixed_envirmap', 160000, 16)
    for k, w in fx["renderer_eval"].items():
        eq(got[k].detach(), w)


def test_init_model_forward(golden_init):
    fx = golden_init
    rgb, dep = O.init_forward(oracle_field(fx, with_mask=False), fx["rays"], True, False, 32)
    eq(rgb.detach(), fx["forward_nomask"][0])
    eq(dep, fx["forward_nomask"][1])
    rgb, dep = O.init_forward(oracle_field(fx), fx["rays"], True, False, 32)
    eq(rgb.detach(), fx["forward_mask"][0])
    eq(dep, fx["forward_mask"][1])


def test_update_alpha_mask(golden_rotated):
    fx = golden_rotated
    f = oracle_field(fx, with_mask=False)
    new_aabb = O.update_alpha_mask(f, (24, 24, 24))
    eq(f.alpha_volume, fx["alpha_volume"])
    eq(new_aabb, fx["new_aabb"])


def test_relight_pass(golden_rotated):
    """Environment_Light tables, background lookup and the per-chunk relighting math of scripts/relight_importance.py
    (with the reference's recorded multinomial indices)."""
    fx = golden_rotated
    f = oracle_field(fx)
    env = O.EnvLight({"sunny": fx["env_rgb"]})
    eq(env.hdr_pdf_sample["sunny"], fx["env_pdf_sample"])
    eq(env.hdr_pdf_return["sunny"], fx["env_pdf_return"])
    eq(env.hdr_dir["sunny"], fx["env_dir"])
    eq(env.get_light("sunny", fx["rays"][:, 3:]), fx["relight_bg_lookup"])
    w, wo = O.relight_chunk(f, env, "sunny", fx["rays"], fx["relight_maps"], 1.7, fx["relight_idx"], 64)
    eq(wo, fx["relight_without_bg"])
    eq(w, fx["relight_with_bg"])
