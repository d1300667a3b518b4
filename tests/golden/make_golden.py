"""Generate golden fixtures by running the REAL reference (a checkout of the original TensoIR project):

    python tests/golden/make_golden.py <path of the original project> [<output directory>]

Writes tests/golden/*.pt: small seeded inputs, the reference model's state_dict / alpha mask,
and the reference's outputs for every hot-path function (SURVEY.md §8a).  The oracle
(oracle/tensoir_oracle.py) is replayed against these in tests/test_oracle_golden.py, and the
CUDA path is checked against the same fixtures in the -m gpu tests.  Also writes the names the
reference's own modules import from ``models.*`` (reference_imports.json) and the reference's
grid_sample outside [-1, 1] (grid_sample_outside.pt), which tests/test_dropin_cpu.py checks
dropin/ against.  No file may exceed 1 MB: the rotated model's state_dict is stored in a file of
its own, and its training gradients as a fixed sample (see ``sample_grads``).
"""
import ast
import json
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(os.path.dirname(HERE))
REF = None          # the original project's checkout, set by main()
sys.path.insert(0, REPO)
GRAD_SAMPLE = 2048  # gradient entries kept per tensor with more entries than this: the largest half + a seeded rest


def import_reference():
    """Put the reference on sys.path with the stubs SURVEY.md §8c lists."""
    kornia = types.ModuleType("kornia")

    def create_meshgrid(h, w, normalized_coordinates=True, device=None, dtype=torch.float32):
        xs = torch.linspace(0, w - 1, w, dtype=dtype)
        ys = torch.linspace(0, h - 1, h, dtype=dtype)
        gy, gx = torch.meshgrid(ys, xs, indexing='ij')
        return torch.stack([gx, gy], -1)[None]

    kornia.create_meshgrid = create_meshgrid
    sys.modules.setdefault("kornia", kornia)
    for name in ("imageio", "lpips", "skimage", "skimage.measure", "plyfile", "configargparse"):
        sys.modules.setdefault(name, types.ModuleType(name))
    if REF not in sys.path:
        sys.path.insert(0, REF)
    import models.relight_utils as ru
    import models.tensoRF_rotated_lights as rot
    import models.tensoRF_general_multi_lights as gen
    import models.tensoRF_init as ini
    orig = ru.sample_ray_equally

    def sample_ray_equally_cpu(tensoIR, rays_o, rays_d, nSample=-1, vis_near=0.03, vis_far=1.5, device=None):
        return orig(tensoIR, rays_o, rays_d, nSample=nSample, vis_near=vis_near, vis_far=vis_far,
                    device=rays_o.device)

    ru.sample_ray_equally = sample_ray_equally_cpu
    return ru, rot, gen, ini


def _args(n=24, near=0.05, far=1.5):
    a = types.SimpleNamespace()
    a.second_nSample, a.second_near, a.second_far = n, near, far
    return a


def build_rotated(rot, G=24, lights=('000', '120'), seed=20211202):
    from tensoir_b200.synthetic import install_lego_density
    torch.manual_seed(seed)
    aabb = torch.tensor([[-1.5, -1.5, -1.5], [1.5, 1.5, 1.5]])
    m = rot.TensorVMSplit(aabb, [G, G, G], 'cpu', density_n_comp=[16, 16, 16], appearance_n_comp=[48, 48, 48],
                          app_dim=27, near_far=[2.0, 6.0], shadingMode='MLP_Fea', alphaMask_thres=0.001,
                          density_shift=-10, distance_scale=25, pos_pe=2, view_pe=2, fea_pe=2, featureC=128,
                          step_ratio=0.5, fea2denseAct='softplus', normals_kind='derived_plus_predicted',
                          light_rotation=list(lights), light_kind='sg', dataset=None, numLgtSGs=128)
    install_lego_density(m)
    return m


def rays_for(n, seed=3):
    from tensoir_b200.synthetic import hemisphere_poses, pixel_rays
    poses = hemisphere_poses(4)
    g = torch.Generator().manual_seed(seed)
    out = []
    for v in range(4):
        pix = torch.randint(0, 800 * 800, (n // 4,), generator=g)
        # bias towards the image centre so most rays hit the object
        j = (400 + (pix // 800 - 400) * 0.45).long()
        i = (400 + (pix % 800 - 400) * 0.45).long()
        out.append(pixel_rays(poses[v], j * 800 + i))
    return torch.cat(out, 0)


def sample_grads(grads, n=GRAD_SAMPLE, seed=5):
    """name -> None or {idx, val, absmax}: every entry of a small gradient; of a larger one the n // 2 entries of
    largest magnitude plus n - n // 2 seeded uniform draws from the rest.  ``absmax`` is the whole tensor's, so a
    relative error keeps the scale of the full comparison."""
    g = torch.Generator().manual_seed(seed)
    out = {}
    for k, w in grads.items():
        if w is None:
            out[k] = None
            continue
        flat = w.reshape(-1)
        if flat.numel() <= n:
            idx = torch.arange(flat.numel())
        else:
            top = flat.abs().topk(n // 2).indices
            rest = torch.ones(flat.numel(), dtype=torch.bool)
            rest[top] = False
            rest = rest.nonzero().reshape(-1)
            idx = torch.cat([top, rest[torch.randperm(rest.numel(), generator=g)[:n - n // 2]]]).sort().values
        out[k] = dict(idx=idx.to(torch.int32), val=flat[idx].clone(), absmax=flat.abs().max().clone())
    return out


def reference_imports():
    """{importer: [[module, [names]]]}: every ``from models.X import a, b`` in the reference outside models/ (the
    modules an unchanged script loads through dropin/).  Star imports name nothing and are left out."""
    out = {}
    for d, _, files in sorted(os.walk(REF)):
        rel = os.path.relpath(d, REF)
        top = rel.split(os.sep)[0]
        if top in ("models", "__pycache__") or (top != "." and top.startswith(".")):
            continue
        for fn in sorted(files):
            if not fn.endswith(".py"):
                continue
            path = os.path.join(d, fn)
            for node in ast.walk(ast.parse(open(path).read(), path)):
                if isinstance(node, ast.ImportFrom) and (node.module or "").startswith("models."):
                    names = [a.name for a in node.names if a.name != "*"]
                    if names:
                        out.setdefault(os.path.relpath(path, REF), []).append([node.module, names])
    return out


def grid_sample_outside(ru):
    """The reference's clamped grid_sample (models/relight_utils.py) on coordinates inside and outside [-1, 1]."""
    g = torch.Generator().manual_seed(0)
    img = torch.randn(2, 5, 7, 9, generator=g)
    grid = torch.rand(2, 6, 4, 2, generator=g) * 3 - 1.5
    return dict(img=img, grid=grid, out=ru.grid_sample(img, grid).detach().clone())


def tolist(t):
    return [x.detach().clone() if torch.is_tensor(x) else x for x in t]


def main():
    global REF, HERE
    if len(sys.argv) < 2:
        raise SystemExit(__doc__)
    REF = os.path.abspath(sys.argv[1])
    if len(sys.argv) > 2:
        HERE = os.path.abspath(sys.argv[2])
        os.makedirs(HERE, exist_ok=True)
    ru, rot, gen, ini = import_reference()
    import renderer as ref_renderer
    out = {}

    # ---------------- rotated multi-light model -----------------------------------------
    m = build_rotated(rot)
    new_aabb = m.updateAlphaMask((24, 24, 24))
    sd = {k: v.detach().clone() for k, v in m.state_dict().items()}
    fx = dict(kind="rotated", state_dict=sd, aabb=m.aabb.clone(), grid_size=m.gridSize.tolist(),
              light_rotation=list(m.light_rotation), alpha_volume=m.alphaMask.alpha_volume.clone(),
              alpha_aabb=m.alphaMask.aabb.clone(), new_aabb=new_aabb.clone(), nSamples=m.nSamples,
              stepSize=float(m.stepSize))
    rays = rays_for(64)
    light_idx = (torch.arange(64) % 2).view(-1, 1).to(torch.int32)
    fx["rays"], fx["light_idx"] = rays, light_idx

    # a) unit functions on random points
    g = torch.Generator().manual_seed(11)
    pts = (torch.rand(257, 3, generator=g) * 2 - 1) * 1.45
    xn = m.normalize_coord(pts)
    fx["pts"] = pts
    fx["sample_alpha"] = m.alphaMask.sample_alpha(pts).clone()
    fx["density_feature"] = m.compute_densityfeature(xn).detach().clone()
    fx["sigma"] = m.feature2density(m.compute_densityfeature(xn)).detach().clone()
    li = (torch.arange(257) % 2).view(-1, 1).to(torch.int32)
    rad, intr = m.compute_bothfeature(xn, li)
    fx["li"], fx["rad_feat"], fx["intr_feat"] = li, rad.detach().clone(), intr.detach().clone()
    fx["app_feat"] = m.compute_appfeature(xn, li).detach().clone()
    fx["intrin_only"] = m.compute_intrinfeature(xn).detach().clone()
    vd = torch.nn.functional.normalize(torch.randn(257, 3, generator=g), dim=-1)
    fx["viewdirs"] = vd
    fx["mlp_rgb"] = m.renderModule(xn, vd, rad).detach().clone()
    fx["mlp_brdf"] = m.renderModule_brdf(xn, intr).detach().clone()
    fx["mlp_normal"] = m.renderModule_normal(xn, intr).detach().clone()
    # jittered points may leave [-1,1]: exercises the clamped sampler (relight_utils.py:57-107)
    xj = (xn + 0.05 * torch.randn(257, 3, generator=g)).detach()
    fx["xj"] = xj
    fx["derived_normals"] = m.compute_derived_normals(xj.clone()).detach().clone()

    # b) sample_ray (eval + train with recorded jitter)
    p, z, v = m.sample_ray(rays[:, :3], rays[:, 3:6], is_train=False, N_samples=-1)
    fx["sample_ray_eval"] = (p.clone(), z.clone(), v.clone())
    torch.manual_seed(5)
    p, z, v = m.sample_ray(rays[:, :3], rays[:, 3:6], is_train=True, N_samples=40)
    torch.manual_seed(5)
    fx["jitter40"] = torch.rand(64, 1)
    fx["sample_ray_train"] = (p.clone(), z.clone(), v.clone())

    # c) secondary marches
    surf = (torch.rand(96, 3, generator=g) * 2 - 1) * torch.tensor([1.0, 1.0, 0.9])
    dirs = torch.nn.functional.normalize(torch.randn(96, 3, generator=g), dim=-1)
    fx["surf"], fx["dirs"] = surf, dirs
    fx["transmittance"] = tolist(ru.compute_transmittance(tensoIR=m, surf_pts=surf, light_in_dir=dirs, nSample=96,
                                                          vis_near=0.05, vis_far=1.5))
    li2 = (torch.arange(96) % 2).view(-1, 1).to(torch.int32)
    fx["li2"] = li2
    fx["radiance"] = tolist(ru.compute_radiance(tensoIR=m, surf_pts=surf, light_in_dir=dirs, light_idx=li2,
                                                nSample=96, vis_near=0.05, vis_far=1.5))

    # d) primary forward, eval (deterministic), relight on/off
    torch.manual_seed(101)   # eval still draws the xyz jitter (tensorBase_rotated_lights.py:937)
    res = m(rays, light_idx, white_bg=True, is_train=False, ndc_ray=False, is_relight=True, N_samples=-1)
    fx["primary_eval"] = tolist(res)
    res = m(rays, light_idx, white_bg=True, is_train=False, ndc_ray=False, is_relight=False, N_samples=-1)
    fx["primary_eval_norelight"] = tolist(res)

    # e) lights / BRDF
    fx["fixed_dirs"] = m.gen_light_incident_dirs(method='fixed_envirmap').clone()
    fx["area_weight"] = m.light_area_weight.clone()
    fx["light_rgbs"] = m.get_light_rgbs(fx["fixed_dirs"], device='cpu').detach().clone()
    nrm = torch.nn.functional.normalize(torch.randn(9, 3, generator=g), dim=-1)
    rough = torch.rand(9, 1, generator=g).repeat(1, 3) * 0.9 + 0.09
    fres = torch.full((9, 3), 0.04)
    v2c = torch.nn.functional.normalize(torch.randn(9, 3, generator=g), dim=-1)
    l2 = fx["fixed_dirs"][None].repeat(9, 1, 1)
    fx["ggx_in"] = (nrm, v2c, rough, fres)
    fx["ggx"] = ru.GGX_specular(nrm, v2c, l2, rough, fres).clone()

    # f) the boundary: eval path (bit-reproducible), then train path with recorded randoms + grads
    args = _args(24)
    torch.manual_seed(102)
    ret = ref_renderer.Renderer_TensoIR_train(rays, None, light_idx, m, N_samples=-1, ndc_ray=False, white_bg=True,
                                              is_train=False, is_relight=True, sample_method='fixed_envirmap',
                                              chunk_size=160000, device='cpu', args=args)
    fx["renderer_eval"] = {k: (v.detach().clone() if torch.is_tensor(v) else v) for k, v in ret.items()}

    torch.manual_seed(77)
    m.zero_grad()
    ret = ref_renderer.Renderer_TensoIR_train(rays, None, light_idx, m, N_samples=60, ndc_ray=False, white_bg=True,
                                              is_train=True, is_relight=True, sample_method='stratified_sampling',
                                              chunk_size=160000, device='cpu', args=args)
    target = torch.full_like(ret["rgb_map"], 0.5)
    loss = (((ret["rgb_map"] - target) ** 2).mean() + 0.2 * ((ret["rgb_with_brdf_map"] - target) ** 2).mean()
            + 0.0005 * ret["normals_diff_map"].mean() + 0.001 * ret["normals_orientation_loss_map"].mean()
            + 0.001 * ret["albedo_smoothness_loss"] + 0.001 * ret["roughness_smoothness_loss"])
    loss.backward()
    fx["renderer_train"] = {k: (v.detach().clone() if torch.is_tensor(v) else v) for k, v in ret.items()}
    fx["renderer_train_loss"] = loss.detach().clone()
    fx["renderer_train_grads"] = {k: (p.grad.detach().clone() if p.grad is not None else None)
                                  for k, p in m.named_parameters()}
    # replay the same random stream to record the draws (order: jitter, xyz noise, bg coin skipped because
    # white_bg short-circuits, light jitter x2)
    torch.manual_seed(77)
    jit = torch.rand(64, 1)
    n_app = int((ret["acc_map"] * 0 + 1).sum() * 0)  # placeholder, real count below
    # count app samples by re-running the primary with the same stream
    torch.manual_seed(77)
    with torch.no_grad():
        xyz, z, valid = m.sample_ray(rays[:, :3], rays[:, 3:6], is_train=True, N_samples=60)
    # number of app samples = rows of the randn draw; recover it by replaying the oracle in the test instead.
    fx["train_seed"] = 77
    fx["train_jitter"] = jit
    # g) relighting pass (scripts/relight_importance.py:99-181) with the reference's Environment_Light on a synthetic
    #    Radiance .hdr (log-normal radiance + a sun disc), multinomial draws recorded
    import cv2, tempfile
    rs = np.random.RandomState(7)
    envmap = np.exp(rs.normal(-1.0, 0.6, size=(16, 32, 3))).astype(np.float32)
    envmap[3:5, 20:22] += 40.0
    tmpd = tempfile.mkdtemp()
    cv2.imwrite(os.path.join(tmpd, "sunny.hdr"), cv2.cvtColor(envmap, cv2.COLOR_RGB2BGR))
    env = ru.Environment_Light(tmpd, device='cpu')
    fx["env_rgb"] = env.hdr_rgbs["sunny"].clone()
    fx["env_pdf_sample"], fx["env_pdf_return"] = env.hdr_pdf_sample["sunny"].clone(), env.hdr_pdf_return["sunny"].clone()
    fx["env_dir"] = env.hdr_dir["sunny"].clone()
    torch.manual_seed(31)
    with torch.enable_grad():
        prim = m(rays, light_idx, is_train=False, white_bg=True, ndc_ray=False, N_samples=-1)
    rgb_c, depth_c, normal_c, albedo_c, rough_c, fresnel_c, acc_c = [t.detach() for t in prim[:7]]
    amask = acc_c > 0.5
    torch.manual_seed(32)
    ldir, lrgb, lpdf = env.sample_light("sunny", int(amask.sum()), 64)
    torch.manual_seed(32)
    fx["relight_idx"] = torch.multinomial(env.hdr_pdf_sample["sunny"].view(-1).expand(int(amask.sum()), -1), 64,
                                          replacement=True)
    surf2c = ru.safe_l2_normalize(-rays[:, 3:][amask], dim=-1)
    cosine = torch.einsum("ijk,ik->ij", ldir, normal_c[amask])
    cmask = cosine > 1e-6
    vis = torch.zeros((*cmask.shape, 1))
    surf = (rays[:, :3] + depth_c.unsqueeze(-1) * rays[:, 3:])[amask]
    nerv, nerf = ru.compute_transmittance(tensoIR=m, surf_pts=surf[:, None, :].expand((*cmask.shape, 3))[cmask],
                                          light_in_dir=ldir[cmask], nSample=96, vis_near=0.05, vis_far=1.5)
    vis[cmask] = nerv.unsqueeze(-1)
    spec = ru.brdf_specular(normal_c[amask], surf2c, ldir, rough_c[amask].repeat(1, 3), fresnel_c[amask])
    brdf = (albedo_c[amask] * 1.7).unsqueeze(1).expand(-1, 64, -1) / np.pi + spec
    srgb = torch.clamp(torch.mean(brdf * (vis * lrgb) * cosine[:, :, None] / lpdf, dim=1), min=0.0, max=1.0)
    srgb = ru.linear2srgb_torch(srgb)
    bg = ru.linear2srgb_torch(torch.clamp(env.get_light("sunny", rays[:, 3:]), min=0.0, max=1.0))
    wo = torch.ones_like(bg)
    wo[amask] = srgb
    acc_t = acc_c[..., None].clone()
    acc_t[acc_t <= 0.9] = 0.0
    fx["relight_maps"] = (depth_c, normal_c, albedo_c, rough_c.repeat(1, 3), fresnel_c, acc_c)
    fx["relight_with_bg"], fx["relight_without_bg"] = acc_t * wo + (1.0 - acc_t) * bg, wo
    fx["relight_bg_lookup"] = env.get_light("sunny", rays[:, 3:]).clone()
    # e2) importance sampling of the SG light (tensorBase_rotated_lights.py:547-572), seeded
    _glr = m.get_light_rgbs          # the reference omits device= on this call (default 'cuda'); pin it to the CPU
    m.get_light_rgbs = lambda dirs=None, device='cpu': _glr(dirs, device='cpu')
    torch.manual_seed(41)
    fx["importance_sample"] = tolist(m.gen_light_incident_dirs(sample_number=64, method='importance_sample',
                                                               device='cpu'))
    del m.get_light_rgbs

    # h) regularisers and grid maintenance (tensoRF_rotated_lights.py:60-92, :226-288) on a fresh copy
    m2 = build_rotated(rot)
    m2.load_state_dict(sd)
    m2.alphaMask = rot.AlphaGridMask('cpu', fx["alpha_aabb"], fx["alpha_volume"])
    from utils import TVLoss
    tv = TVLoss()
    fx["reg"] = dict(ortho=m2.vector_comp_diffs().detach().clone(), l1=m2.density_L1().detach().clone(),
                     tv_density=m2.TV_loss_density(tv).detach().clone(), tv_app=m2.TV_loss_app(tv).detach().clone())
    m2.shrink(new_aabb.clone())
    fx["shrink"] = dict(aabb=m2.aabb.clone(), grid=m2.gridSize.tolist(), nSamples=m2.nSamples,
                        density_plane0=m2.density_plane[0].detach().clone(), app_line2=m2.app_line[2].detach().clone())
    m2.upsample_volume_grid([30, 31, 29])
    fx["upsample"] = dict(grid=m2.gridSize.tolist(), nSamples=m2.nSamples, stepSize=float(m2.stepSize),
                          density_plane1=m2.density_plane[1].detach().clone(),
                          app_line0=m2.app_line[0].detach().clone())
    out["rotated"] = fx
    torch.save(fx.pop("state_dict"), os.path.join(HERE, "rotated_g24_state.pt"))
    fx["state_dict"] = "rotated_g24_state.pt"          # resolved by tests/gpu_helpers.load_fixture
    fx["renderer_train_grads_sample"] = sample_grads(fx.pop("renderer_train_grads"))
    torch.save(fx, os.path.join(HERE, "rotated_g24.pt"))

    # ---------------- general multi-light model (boundary smoke) -------------------------
    from tensoir_b200.synthetic import install_lego_density
    torch.manual_seed(20211202)
    aabb = torch.tensor([[-1.5, -1.5, -1.5], [1.5, 1.5, 1.5]])
    mg = gen.TensorVMSplit(aabb, [20, 20, 20], 'cpu', density_n_comp=[16, 16, 16], appearance_n_comp=[48, 48, 48],
                           app_dim=27, near_far=[2.0, 6.0], shadingMode='MLP_Fea', alphaMask_thres=0.001,
                           density_shift=-10, distance_scale=25, pos_pe=2, view_pe=2, fea_pe=2, featureC=128,
                           step_ratio=0.5, fea2denseAct='softplus', normals_kind='derived_plus_predicted',
                           light_name_list=['sunset', 'snow', 'courtyard'], light_kind='sg', dataset=None,
                           numLgtSGs=128)
    install_lego_density(mg)
    mg.updateAlphaMask((20, 20, 20))
    rays_g = rays_for(32, seed=9)
    lig = (torch.arange(32) % 3).view(-1, 1).to(torch.int32)
    torch.manual_seed(103)
    ret = ref_renderer.Renderer_TensoIR_train(rays_g, None, lig, mg, N_samples=-1, ndc_ray=False, white_bg=True,
                                              is_train=False, is_relight=True, sample_method='fixed_envirmap',
                                              chunk_size=160000, device='cpu', args=_args(16))
    fg = dict(kind="general", state_dict={k: v.detach().clone() for k, v in mg.state_dict().items()},
              lgt_sgs_list=[p.detach().clone() for p in mg.lgtSGs_list], aabb=mg.aabb.clone(),
              grid_size=mg.gridSize.tolist(), alpha_volume=mg.alphaMask.alpha_volume.clone(),
              alpha_aabb=mg.alphaMask.aabb.clone(), rays=rays_g, light_idx=lig,
              renderer_eval={k: (v.detach().clone() if torch.is_tensor(v) else v) for k, v in ret.items()})
    torch.save(fg, os.path.join(HERE, "general_g20.pt"))

    # ---------------- tensoRF_init model (BASELINE config 1 semantics) -------------------
    torch.manual_seed(20211202)
    mi = ini.TensorVMSplit(aabb, [24, 24, 24], 'cpu', density_n_comp=[16, 16, 16], appearance_n_comp=[48, 48, 48],
                           app_dim=27, near_far=[2.0, 6.0], shadingMode='MLP_Fea', alphaMask_thres=0.001,
                           density_shift=-10, distance_scale=25, pos_pe=2, view_pe=2, fea_pe=2, featureC=128,
                           step_ratio=0.5, fea2denseAct='softplus')
    install_lego_density(mi)
    rays_i = rays_for(64, seed=21)
    rgb0, dep0 = mi(rays_i, white_bg=True, is_train=False, ndc_ray=False, N_samples=32)   # no alpha mask yet
    mi.updateAlphaMask((24, 24, 24))
    rgb1, dep1 = mi(rays_i, white_bg=True, is_train=False, ndc_ray=False, N_samples=32)
    fi = dict(kind="init", state_dict={k: v.detach().clone() for k, v in mi.state_dict().items()},
              aabb=mi.aabb.clone(), grid_size=mi.gridSize.tolist(), alpha_volume=mi.alphaMask.alpha_volume.clone(),
              alpha_aabb=mi.alphaMask.aabb.clone(), rays=rays_i,
              forward_nomask=(rgb0.detach().clone(), dep0.detach().clone()),
              forward_mask=(rgb1.detach().clone(), dep1.detach().clone()))
    torch.save(fi, os.path.join(HERE, "init_g24.pt"))
    torch.save(grid_sample_outside(ru), os.path.join(HERE, "grid_sample_outside.pt"))
    with open(os.path.join(HERE, "reference_imports.json"), "w") as fh:
        json.dump(reference_imports(), fh, indent=1, sort_keys=True)
        fh.write("\n")
    for n in ("rotated_g24.pt", "rotated_g24_state.pt", "general_g20.pt", "init_g24.pt", "grid_sample_outside.pt"):
        print(n, os.path.getsize(os.path.join(HERE, n)) // 1024, "KiB")


if __name__ == "__main__":
    main()
