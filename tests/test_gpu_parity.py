"""GPU parity: the CUDA path (through the C ABI) vs the reference-generated golden fixtures and the oracle.

Tolerances: fp32 path, north-star bar 1e-4 relative on rendered maps.  Counts (mask / density / app samples)
must match the oracle exactly on these fixtures."""
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import tensoir_oracle as O            # noqa: E402
from helpers import oracle_field, named_oracle_params   # noqa: E402
from gpu_helpers import model_from_fixture, renderer_args   # noqa: E402

DEV = "cuda:0"
TOL = 1e-4


def close(got, want, tol=TOL, what=""):
    got = got.detach().float().cpu()
    want = want.detach().float().cpu()
    assert got.shape == want.shape, (what, got.shape, want.shape)
    err = (got - want).abs()
    bound = tol * (1.0 + want.abs())
    assert bool((err <= bound).all()), (what, float(err.max()), float((err / bound).max()))


def psnr(got, want):
    mse = ((got.detach().float().cpu() - want.detach().float().cpu()) ** 2).mean()
    return float(-10.0 * torch.log10(mse.clamp_min(1e-20)))


@pytest.fixture(scope="module")
def rot(golden_rotated):
    from tensoir_b200 import _lib
    _lib.load()
    return golden_rotated, model_from_fixture(golden_rotated, DEV)


def test_unit_kernels(rot):
    from tensoir_b200 import ops
    fx, m = rot
    pts = fx["pts"].to(DEV)
    xn = m.normalize_coord(pts)
    assert torch.equal(ops.alpha_mask_points(m, pts).cpu(), fx["sample_alpha"] > 0)
    feat, sig = ops.density_points(m, xn)
    close(feat, fx["density_feature"], 2e-5, "density_feature")
    close(sig, fx["sigma"], 2e-5, "sigma")
    close(m.compute_densityfeature(xn), fx["density_feature"], 2e-5)
    li = fx["li"].to(DEV)
    rad, intr = m.compute_bothfeature(xn, li)
    close(rad, fx["rad_feat"], 2e-5, "rad")
    close(intr, fx["intr_feat"], 2e-5, "intr")
    close(m.compute_appfeature(xn, li), fx["app_feat"], 2e-5)
    close(m.compute_intrinfeature(xn), fx["intrin_only"], 2e-5)
    vd = fx["viewdirs"].to(DEV)
    close(ops.app_mlp_points(m, xn, vd, li, head="renderModule"), fx["mlp_rgb"], 5e-5, "mlp_rgb")
    close(ops.app_mlp_points(m, xn, xn, None, head="renderModule_brdf", light="mean"), fx["mlp_brdf"], 5e-5, "brdf")
    close(ops.app_mlp_points(m, xn, xn, None, head="renderModule_normal", light="mean"), fx["mlp_normal"], 5e-5, "nrm")
    # derived normals: compare the raw gradient (absolute, vs its scale) and the unit normals where the gradient
    # is well conditioned (a normalised ~0 gradient amplifies summation-order noise by up to 1e6)
    from tensoir_b200.primary import _derived_normals
    from tensoir_b200 import vm_autograd as vm
    f = oracle_field(fx)
    xj = fx["xj"].clone().requires_grad_(True)
    sig = O.feature2density(f, O.density_feature_with_xyz_grad(f, xj))
    g_ref = torch.autograd.grad(sig.sum(), xj)[0]
    ft, dfdx = vm.density_feature_and_grad(m, fx["xj"].to(DEV))
    g_got = (torch.sigmoid(ft - 10)[:, None] * dfdx).cpu()
    assert float((g_got - g_ref).detach().abs().max()) < 1e-4 * float(g_ref.abs().max())
    well = g_ref.norm(dim=-1) > 1e-3 * float(g_ref.norm(dim=-1).max())
    assert int(well.sum()) > 20
    close(_derived_normals(m, fx["xj"].to(DEV))[well.to(DEV)], fx["derived_normals"][well], 5e-4, "derived_normals")


def test_valid_sample_lists_bit_exact(rot):
    """sample_ray + bbox + alpha-mask filter: indices must equal the reference's masks exactly."""
    from tensoir_b200 import vm_autograd as vm
    fx, m = rot
    f = oracle_field(fx)
    rays = fx["rays"]
    for is_train, ns, jit in ((False, -1, None), (True, 40, fx["jitter40"])):
        pts, z, valid = O.sample_ray(f, rays[:, :3], rays[:, 3:6], is_train, ns, jitter=jit)
        valid = O._refine_valid(f, pts, valid)
        lst = vm.valid_samples(m, rays[:, :3].to(DEV), rays[:, 3:6].to(DEV), n_samples=ns,
                               jitter=None if jit is None else jit.to(DEV))
        idx = valid.nonzero()
        assert torch.equal(lst["ray"].cpu().long(), idx[:, 0])
        assert torch.equal(lst["sample"].cpu().long(), idx[:, 1])
        assert torch.equal(lst["z"].cpu(), z.expand(valid.shape)[valid])
        assert torch.equal(lst["xn"].cpu(), O.normalize_coord(f, pts)[valid])


def test_secondary_marches(rot):
    from tensoir_b200 import ops, relight_utils as RU
    fx, m = rot
    f = oracle_field(fx)
    surf, dirs, li2 = fx["surf"].to(DEV), fx["dirs"].to(DEV), fx["li2"].to(DEV)
    cnt = ops.new_counters(DEV)
    m.__dict__["_tir_counters"] = cnt
    nerv, nerf = RU.compute_transmittance(m, surf, dirs, nSample=96, vis_near=0.05, vis_far=1.5)
    close(nerv, fx["transmittance"][0], 2e-5, "nerv_vis")
    close(nerf, fx["transmittance"][1], 2e-5, "nerfactor_vis")
    O.compute_transmittance(f, fx["surf"], fx["dirs"], 96, 0.05, 1.5)
    c = ops.counters_dict(cnt)
    assert c["density"] == f.counters["density"] and c["mask"] == f.counters["mask"]
    cnt.zero_()
    f.counters.clear()
    nerv, nerf, ind = RU.compute_radiance(m, surf, dirs, li2, nSample=96, vis_near=0.05, vis_far=1.5)
    close(nerv, fx["radiance"][0], 2e-5)
    close(nerf, fx["radiance"][1], 2e-5)
    close(ind, fx["radiance"][2], TOL, "indirect")
    *_, valid, app_mask, weight = O.compute_radiance(f, fx["surf"], fx["dirs"], fx["li2"], 96, 0.05, 1.5,
                                                     return_aux=True)
    c = ops.counters_dict(cnt)
    assert c["overflow"] == 0
    assert (c["mask"], c["density"], c["app"]) == (f.counters["mask"], f.counters["density"], f.counters["app"])
    # the compacted sample list holds exactly the reference's app_mask indices
    sm = m.__dict__["_tir_scratch"].samples()
    key = (sm["ray"].long() * 96 + sm["sample"].long()).cpu().sort().values
    want = app_mask.nonzero()
    assert torch.equal(key, (want[:, 0] * 96 + want[:, 1]).sort().values)
    del m.__dict__["_tir_counters"]


def test_dense_secondary_vs_explicit(rot):
    """tir_secondary_radiance (rays generated on chip) == compute_radiance on the expanded ray list."""
    from tensoir_b200 import ops
    fx, m = rot
    f = oracle_field(fx)
    g = torch.Generator().manual_seed(4)
    pts = (torch.rand(7, 3, generator=g) * 2 - 1) * 0.9
    nrm = torch.nn.functional.normalize(torch.randn(7, 3, generator=g), dim=-1)
    li = (torch.arange(7) % 2).view(-1, 1).to(torch.int32)
    dirs = fx["fixed_dirs"]
    vis, ind, _ = ops.secondary_radiance(m, pts.to(DEV), nrm.to(DEV), li.to(DEV), dirs.to(DEV), n_sample=24)
    cos = torch.clamp(torch.einsum("jk,ik->ij", dirs, nrm), min=0)
    mask = cos > 1e-6
    P = pts[:, None, :].expand(-1, dirs.shape[0], -1)[mask]
    D = dirs[None].expand(7, -1, -1)[mask]
    L = li.view(-1, 1, 1).expand(-1, dirs.shape[0], 1)[mask]
    v, _, i = O.compute_radiance(f, P, D, L, 24, 0.05, 1.5)
    want_v = torch.zeros(7, dirs.shape[0], 1)
    want_i = torch.zeros(7, dirs.shape[0], 3)
    want_v[mask] = v[:, None]
    want_i[mask] = i
    close(vis, want_v, 2e-5, "vis")
    close(ind, want_i, TOL, "indirect")


def test_primary_eval(rot):
    fx, m = rot
    rays, li = fx["rays"].to(DEV), fx["light_idx"].to(DEV)
    torch.manual_seed(101)
    m.__dict__["_tir_randn_like"] = lambda t: torch.randn(t.shape).to(t.device)
    with torch.no_grad():
        got = m(rays, li, white_bg=True, is_train=False, is_relight=True, N_samples=-1)
    names = ["rgb", "depth", "normal", "albedo", "rough", "fresnel", "acc", "ndiff", "norient", "acc_mask",
             "alb_loss", "rough_loss"]
    for n, g, w in zip(names, got, fx["primary_eval"]):
        if w.dtype == torch.bool:
            assert torch.equal(g.cpu(), w), n
        else:
            close(g, w, TOL, n)
    with torch.no_grad():
        got = m(rays, li, white_bg=True, is_train=False, is_relight=False, N_samples=-1)
    for n, g, w in zip(names, got, fx["primary_eval_norelight"]):
        if w is None:
            assert g is None
        else:
            close(g, w, TOL, n)
    del m.__dict__["_tir_randn_like"]


def test_boundary_eval(rot):
    from tensoir_b200 import Renderer_TensoIR_train
    fx, m = rot
    torch.manual_seed(102)
    m.__dict__["_tir_randn_like"] = lambda t: torch.randn(t.shape).to(t.device)
    with torch.no_grad():
        got = Renderer_TensoIR_train(fx["rays"], None, fx["light_idx"], m, N_samples=-1, white_bg=True,
                                     is_train=False, is_relight=True, sample_method='fixed_envirmap',
                                     chunk_size=160000, device=DEV, args=renderer_args(24))
    for k, w in fx["renderer_eval"].items():
        close(got[k], w, TOL, k)
    # BASELINE metric, second half: PSNR of our images against the reference's (1e-4 parity => well above 70 dB)
    for k in ("rgb_map", "rgb_with_brdf_map"):
        assert psnr(got[k], fx["renderer_eval"][k]) > 70.0, k
    del m.__dict__["_tir_randn_like"]


def test_boundary_train_step_grads(golden_rotated):
    """Full training-mode boundary + backward: outputs, loss and every parameter gradient vs the reference."""
    from tensoir_b200 import Renderer_TensoIR_train
    fx = golden_rotated
    m = model_from_fixture(fx, DEV)
    m.__dict__["_tir_randn_like"] = lambda t: torch.randn(t.shape).to(t.device)   # CPU stream like the oracle run
    torch.manual_seed(fx["train_seed"])
    got = Renderer_TensoIR_train(fx["rays"], None, fx["light_idx"], m, N_samples=60, white_bg=True, is_train=True,
                                 is_relight=True, sample_method='stratified_sampling', chunk_size=160000,
                                 device=DEV, args=renderer_args(24))
    for k, w in fx["renderer_train"].items():
        close(got[k], w, TOL, k)
    target = torch.full_like(got["rgb_map"], 0.5)
    loss = (((got["rgb_map"] - target) ** 2).mean() + 0.2 * ((got["rgb_with_brdf_map"] - target) ** 2).mean()
            + 0.0005 * got["normals_diff_map"].mean() + 0.001 * got["normals_orientation_loss_map"].mean()
            + 0.001 * got["albedo_smoothness_loss"] + 0.001 * got["roughness_smoothness_loss"])
    loss.backward()
    close(loss, fx["renderer_train_loss"], TOL, "loss")
    n, worst = 0, {}
    for k, p in m.named_parameters():
        w = fx["renderer_train_grads_sample"][k]
        if w is None:
            assert p.grad is None or float(p.grad.abs().max()) == 0.0, k
            continue
        g = p.grad.detach().cpu().reshape(-1)
        scale = float(w["absmax"]) + 1e-12
        err = max(float((g[w["idx"].long()] - w["val"]).abs().max()), abs(float(g.abs().max()) - float(w["absmax"])))
        err /= scale
        worst[k] = err
        n += 1
    assert n >= 20
    bad = {k: v for k, v in worst.items() if v > 5e-4}
    assert not bad, (bad, max(worst.values()))


def test_general_and_init_models(golden_general, golden_init):
    from tensoir_b200 import Renderer_TensoIR_train, OctreeRender_trilinear_fast
    fx = golden_general
    m = model_from_fixture(fx, DEV)
    torch.manual_seed(103)
    m.__dict__["_tir_randn_like"] = lambda t: torch.randn(t.shape).to(t.device)
    with torch.no_grad():
        got = Renderer_TensoIR_train(fx["rays"], None, fx["light_idx"], m, N_samples=-1, white_bg=True,
                                     is_train=False, is_relight=True, sample_method='fixed_envirmap',
                                     chunk_size=160000, device=DEV, args=renderer_args(16))
    for k, w in fx["renderer_eval"].items():
        close(got[k], w, TOL, k)
    fx = golden_init
    for with_mask, key in ((False, "forward_nomask"), (True, "forward_mask")):
        mi = model_from_fixture(fx, DEV, with_mask=with_mask)
        with torch.no_grad():
            rgb, _, depth, _, _ = OctreeRender_trilinear_fast(fx["rays"], mi, chunk=40, N_samples=32, white_bg=True,
                                                              is_train=False, device=DEV)
        close(rgb, fx[key][0], TOL, "rgb")
        close(depth, fx[key][1], TOL, "depth")


def test_update_alpha_mask_and_filtering(golden_rotated):
    fx = golden_rotated
    m = model_from_fixture(fx, DEV, with_mask=False)
    new_aabb = m.updateAlphaMask((24, 24, 24))
    assert torch.equal(m.alphaMask.alpha_volume.cpu(), fx["alpha_volume"])
    close(new_aabb, fx["new_aabb"], 1e-6)
    rays = fx["rays"]
    kept, mask = m.filtering_rays(rays, bbox_only=True)
    assert kept.shape[0] == int(mask.sum())
    f = oracle_field(fx)
    pts, _, _ = O.sample_ray(f, rays[:, :3], rays[:, 3:6], False, 256)
    want = (O.sample_alpha(f, pts.reshape(-1, 3)).view(pts.shape[:-1]) > 0).any(-1)
    _, mask2 = m.filtering_rays(rays, N_samples=256)
    assert torch.equal(mask2, want)


def test_full_size_properties():
    """BASELINE-size checks through size-independent properties: 128^3 lego scene, 4096-ray batch.
    (i) T_last * prod == consistency: nerv_vis in [0,1], nerfactor_vis = 1 - acc; (ii) chunking invariance:
    marching the batch in two halves gives the same per-ray results bit-for-bit; (iii) counters add up."""
    from tensoir_b200 import TensorVMSplit, ops
    from tensoir_b200.synthetic import install_lego_density, hemisphere_poses, training_batch
    torch.manual_seed(20211202)
    aabb = torch.tensor([[-1.5] * 3, [1.5] * 3], device=DEV)
    m = TensorVMSplit(aabb, [128] * 3, DEV, density_n_comp=[16] * 3, appearance_n_comp=[48] * 3, app_dim=27,
                      shadingMode='MLP_Fea', step_ratio=0.5, normals_kind='derived_plus_predicted',
                      light_rotation=['000'], light_kind='sg', alphaMask_thres=0.001)
    install_lego_density(m)
    m.updateAlphaMask((128, 128, 128))
    rays, _ = training_batch(hemisphere_poses(100), 4096, 0)
    rays = rays.to(DEV)
    cnt = ops.new_counters(DEV)
    t, acc, dep = ops.march_density(m, rays[:, :3], rays[:, 3:], n_samples=443, counters=cnt)
    assert float(t.min()) >= 0 and float(t.max()) <= 1 + 1e-6 and float(acc.max()) <= 1 + 1e-5
    t1, a1, d1 = ops.march_density(m, rays[:2048, :3], rays[:2048, 3:], n_samples=443)
    t2, a2, d2 = ops.march_density(m, rays[2048:, :3], rays[2048:, 3:], n_samples=443)
    # chunking invariance (batches of the gather are shared across consecutive rays, so the scan association - not
    # the math - depends on the neighbours: equal to fp32 round-off, not bit-for-bit)
    close(torch.cat([t1, t2]), t, 2e-6, "T chunking")
    close(torch.cat([a1, a2]), acc, 2e-6, "acc chunking")
    close(torch.cat([d1, d2]), dep, 2e-6, "depth chunking")
    c = ops.counters_dict(cnt)
    assert c["rays"] == 4096 and 0 < c["density"] <= c["mask"] <= 4096 * 443
    hit = acc > 0.5
    assert 0.05 < float(hit.float().mean()) < 0.95
    # telescoping identity of raw2alpha: sum_i alpha_i T_i = 1 - prod_i (1 - alpha_i)  =>  acc + T_last = 1
    close(acc + t, torch.ones_like(t), 1e-5, "acc + T_last")
    assert float(dep[hit].min()) > 2.0 and float(dep[hit].max()) < 6.0


def _train_loss(got):
    target = torch.full_like(got["rgb_map"], 0.5)
    return (((got["rgb_map"] - target) ** 2).mean() + 0.2 * ((got["rgb_with_brdf_map"] - target) ** 2).mean()
            + 0.0005 * got["normals_diff_map"].mean() + 0.001 * got["normals_orientation_loss_map"].mean()
            + 0.001 * got["albedo_smoothness_loss"] + 0.001 * got["roughness_smoothness_loss"])


def test_static_capacity_mode_matches_dynamic(golden_rotated):
    """The shape-static form used under CUDA-graph capture (padded lists, no acc_mask compaction) gives the same maps
    and gradients as the dynamic path for identical random inputs."""
    from tensoir_b200 import Renderer_TensoIR_train
    fx = golden_rotated
    rays, li = fx["rays"].to(DEV), fx["light_idx"].to(DEV)
    noise = lambda t: torch.sin(t * 977.0)          # deterministic per row, independent of padding
    outs = []
    for static in (False, True):
        m = model_from_fixture(fx, DEV)
        m.__dict__["_tir_randn_like"] = noise
        torch.manual_seed(5)
        if static:
            jit = torch.rand(64, 1)
            dirs = m.gen_light_incident_dirs(method='stratified_sampling')
            m.__dict__["_tir_static"] = {"cap_valid": 64 * 60, "cap_app": 1024, "jitter": jit.to(DEV),
                                         "dirs": dirs.to(DEV), "overflow": torch.zeros((), dtype=torch.int64, device=DEV),
                                         "stats": torch.zeros(4, dtype=torch.int64, device=DEV),
                                         "overflow_step": torch.zeros((), dtype=torch.int64, device=DEV)}
        got = Renderer_TensoIR_train(rays, None, li, m, N_samples=60, white_bg=True, is_train=True, is_relight=True,
                                     sample_method='stratified_sampling', device=DEV, args=renderer_args(24))
        loss = _train_loss(got)
        loss.backward()
        if static:
            assert int(m.__dict__["_tir_static"]["overflow_step"]) == 0
            assert int(m.__dict__["_tir_static"]["stats"][0]) > 0          # real list lengths are recorded
        outs.append((got, loss, {k: p.grad.detach().clone() for k, p in m.named_parameters() if p.grad is not None}))
    (g0, l0, gr0), (g1, l1, gr1) = outs
    for k in g0:
        close(g1[k], g0[k], 2e-5, k)
    close(l1, l0, 2e-5, "loss")
    assert set(gr0) == set(gr1)
    for k in gr0:
        scale = float(gr0[k].abs().max()) + 1e-12
        assert float((gr0[k] - gr1[k]).abs().max()) / scale < 1e-3, k


def test_cuda_graph_step(golden_rotated):
    """Whole-step capture: replays run, stay finite, never overflow, move the parameters, and the captured loss of the
    first replay equals the eager static step on the same inputs (up to the xyz-noise stream, weight 1e-3)."""
    from tensoir_b200.static_step import StaticTrainStep
    fx = golden_rotated
    m = model_from_fixture(fx, DEV)
    opt = torch.optim.Adam(m.get_optparam_groups(0.02, 0.001), betas=(0.9, 0.99), fused=True, capturable=True)
    rays, li = fx["rays"].to(DEV), fx["light_idx"].to(DEV)
    # the loss also touches parameters directly (L1 regulariser, train_tensoIR.py:271-273): a second gradient producer
    st = StaticTrainStep(m, opt, 64, 60, renderer_args(24), lambda ret, mm: _train_loss(ret) + 4e-5 * mm.density_L1(),
                         device=DEV)
    st.calibrate([(rays, li)])
    before = m.density_plane[0].detach().clone()
    st.capture(warmup=2)
    assert torch.equal(m.density_plane[0].detach(), before)        # capture()'s warm-up executions do not train
    losses = [float(st.run(rays, li)) for _ in range(4)]
    st.flush()
    assert all(l == l and l < 10 for l in losses), losses
    assert st.overflowed() == 0 and st.redone == 0
    assert float((m.density_plane[0] - before).abs().max()) > 0
    assert losses[-1] < losses[0] + 0.05          # Adam on a fixed batch does not diverge
    st.release()


def test_cuda_graph_step_overflow_is_redone(golden_rotated):
    """Lists that are too short never change the computation: the overflowed replay leaves parameters and Adam state
    untouched (found_inf), the host grows the lists, re-captures and redoes the batch; the result equals a run whose
    lists were large enough from the start (up to atomics order / the padded xyz-noise stream)."""
    from tensoir_b200.static_step import StaticTrainStep
    fx = golden_rotated
    rays, li = fx["rays"].to(DEV), fx["light_idx"].to(DEV)
    outs = []
    for tiny in (False, True):
        m = model_from_fixture(fx, DEV)
        m.__dict__["_tir_randn_like"] = lambda t: torch.sin(t * 977.0)      # noise independent of the padding
        opt = torch.optim.Adam(m.get_optparam_groups(0.02, 0.001), betas=(0.9, 0.99), fused=True, capturable=True)
        st = StaticTrainStep(m, opt, 64, 60, renderer_args(24), lambda ret, mm: _train_loss(ret), device=DEV, lag=1)
        st.calibrate([(rays, li)])
        fixed_dirs = m.gen_light_incident_dirs(method='fixed_envirmap')

        def stage(slot, st=st, fixed_dirs=fixed_dirs):       # identical host "randoms" in both runs and in the redo
            st.static["jitter"].fill_(0.5)
            st.static["dirs"].copy_(fixed_dirs)
        st._stage_host_randoms = stage
        if tiny:
            st._set_caps(max(64, st.static["cap_valid"] // 8), max(16, st.static["cap_app"] // 8), 4)
        st.capture(warmup=1)
        torch.manual_seed(5)
        for _ in range(3):
            st.run(rays, li)
        st.flush()
        if tiny:
            assert st.redone >= 1 and st.recaptures >= 1
        else:
            assert st.redone == 0 and st.overflowed() == 0
        steps = {int(v["step"].item()) for v in opt.state.values()}
        assert steps == {3}, steps                        # no-op replays did not advance Adam's step counters
        outs.append((m.renderModule.mlp[0].weight.detach().clone(), m.density_plane[0].detach().clone()))
        st.release()
    (w0, d0), (w1, d1) = outs
    assert float((w0 - w1).abs().max()) < 2e-2 * float(w0.abs().max())
    assert float((d0 - d1).abs().max()) < 2e-2 * max(float(d0.abs().max()), 1e-3)


def test_edge_cases(golden_rotated):
    """Empty and degenerate inputs the reference handles: no rays, rays that miss the aabb entirely (no valid sample,
    no surface hit -> empty secondary batch), zero direction components (sample_ray's 1e-6 substitution,
    tensorBase:709), no alpha mask, a single sample per ray."""
    from tensoir_b200 import Renderer_TensoIR_train, relight_utils as RU, ops
    fx = golden_rotated
    m = model_from_fixture(fx, DEV)
    f = oracle_field(fx)
    args = renderer_args(24)
    # (i) zero rays
    with torch.no_grad():
        out = Renderer_TensoIR_train(torch.zeros(0, 6), None, torch.zeros(0, 1, dtype=torch.int32), m, N_samples=-1,
                                     is_train=False, is_relight=True, device=DEV, args=args)
    assert out["rgb_map"].shape == (0, 3) and out["rgb_with_brdf_map"].shape == (0, 3)
    nv, nf = RU.compute_transmittance(m, torch.zeros(0, 3, device=DEV), torch.zeros(0, 3, device=DEV), 96, 0.05, 1.5)
    assert nv.numel() == 0 and nf.numel() == 0
    # (ii) rays pointing away from the scene + axis-aligned rays with exact zeros in the direction
    o = torch.tensor([[0., 0., 4.], [0., 0., 4.], [4., 0.2, 0.1], [0.3, -4., 0.2]])
    d = torch.tensor([[0., 0., 1.], [0., 0., -1.], [-1., 0., 0.], [0., 1., 0.]])
    rays = torch.cat([o, d], 1)
    li = torch.zeros(4, 1, dtype=torch.int32)
    torch.manual_seed(9)
    m.__dict__["_tir_randn_like"] = lambda t: torch.randn(t.shape).to(t.device)
    with torch.no_grad():
        got = Renderer_TensoIR_train(rays, None, li, m, N_samples=-1, is_train=False, is_relight=True, device=DEV,
                                     args=args)
    torch.manual_seed(9)
    want = O.renderer_train(f, rays, li, -1, True, False, True, 'fixed_envirmap', 160000, 24)
    for k, w in want.items():
        close(got[k], w, TOL, k)
    assert float(got["acc_map"][0]) == 0.0            # the ray that leaves the scene composites nothing
    # (ii-b) a chunk in which EVERY ray misses the aabb (image corners of a full-view render): no valid sample at all
    away = torch.cat([o[:1].repeat(5, 1), d[:1].repeat(5, 1)], 1)
    with torch.no_grad():
        g2 = Renderer_TensoIR_train(away, None, torch.zeros(5, 1, dtype=torch.int32), m, N_samples=-1,
                                    is_train=False, is_relight=True, device=DEV, args=args)
    assert torch.equal(g2["acc_map"].cpu(), torch.zeros(5)) and torch.equal(g2["rgb_with_brdf_map"].cpu(),
                                                                            torch.ones(5, 3))
    # (iii) no alpha mask, one sample per ray
    m2 = model_from_fixture(fx, DEV, with_mask=False)
    f2 = oracle_field(fx, with_mask=False)
    r = fx["rays"][:16]
    t, a, dep = ops.march_density(m2, r[:, :3].to(DEV), r[:, 3:].to(DEV), n_samples=1)
    pts, z, valid = O.sample_ray(f2, r[:, :3], r[:, 3:6], False, 1)
    assert torch.equal(a.cpu(), torch.zeros(16))       # a single sample has dist 0 -> alpha 0 (tensorBase:887)
    t, a, dep = ops.march_density(m2, r[:, :3].to(DEV), r[:, 3:].to(DEV), n_samples=50)
    _, w, tl = O.raw2alpha(*_oracle_sigma_dist(f2, r, 50))
    close(a, w.sum(-1), 2e-5, "acc no-mask")
    close(t, tl.squeeze(-1), 2e-5, "T no-mask")


def _oracle_sigma_dist(f, rays, n):
    pts, z, valid = O.sample_ray(f, rays[:, :3], rays[:, 3:6], False, n)
    dists = torch.cat((z[:, 1:] - z[:, :-1], torch.zeros_like(z[:, :1])), dim=-1).expand(pts.shape[:-1])
    sigma = torch.zeros(pts.shape[:-1])
    xn = O.normalize_coord(f, pts)
    sigma[valid] = O.feature2density(f, O.density_feature(f, xn[valid]))
    return sigma, dists * f.distance_scale


def test_fused_shade_kernel_vs_reference_math(golden_rotated):
    """tir_shade_fwd/_bwd vs the reference's GGX + quadrature expressed in torch (the oracle's functions run on the
    GPU) incl. every input gradient."""
    from tensoir_b200.shade import shade
    f = oracle_field(golden_rotated)
    g = torch.Generator().manual_seed(3)
    bs, nl, L = 37, 512, 2
    nrm = torch.nn.functional.normalize(torch.randn(bs, 3, generator=g), dim=-1)
    # roughness >= 0.25: below that GGX's nom0 = NoH^2 (alpha^2 - 1) + 1 cancels catastrophically near the specular
    # peak and ANY two fp32 evaluation orders (also the reference's own CPU vs GPU) differ by ~1e-3 relative
    alb, rough, fres = torch.rand(bs, 3, generator=g), torch.rand(bs, 1, generator=g).repeat(1, 3) * 0.74 + 0.25, \
        torch.rand(bs, 3, generator=g) * 0.5
    view = torch.nn.functional.normalize(torch.randn(bs, 3, generator=g), dim=-1)
    direct = torch.rand(L, nl, 3, generator=g) * 2
    vis, ind = torch.rand(bs, nl, 1, generator=g), torch.rand(bs, nl, 3, generator=g) * 0.3
    li = (torch.arange(bs) % L).view(-1, 1)
    torch.manual_seed(1)
    dirs = O.gen_light_incident_dirs(f, 'stratified_sampling')
    w = O.generate_envir_map_dir(16, 32)[0]
    leaves = [t.clone().to(DEV).requires_grad_(True) for t in (nrm, alb, rough, fres, direct)]
    leaves_ref = [t.clone().to(DEV).requires_grad_(True) for t in (nrm, alb, rough, fres, direct)]
    cst = [t.to(DEV) for t in (view, li, dirs, w, vis, ind)]
    got = shade(*leaves, cst[0], cst[1], cst[2], cst[3], cst[4], cst[5])
    n_, a_, r_, f_, d_ = leaves_ref
    surf2l = cst[2][None].expand(bs, -1, -1)
    cos = torch.clamp(torch.einsum("ijk,ik->ij", surf2l, n_), min=0.0)
    spec = O.ggx_specular(n_, cst[0], surf2l, r_, f_)
    brdf = a_.unsqueeze(1) / torch.pi + spec
    light = cst[4] * torch.index_select(d_, 0, cst[1].reshape(-1)) + cst[5]
    want = torch.sum(brdf * light * cos[:, :, None] * cst[3][None, :, None], dim=1)
    close(got, want, 5e-5, "shade fwd")
    gw = torch.randn(bs, 3, generator=g).to(DEV)
    (got * gw).sum().backward()
    (want * gw).sum().backward()
    for name, a, b in zip(("normal", "albedo", "rough", "fresnel", "direct"), leaves, leaves_ref):
        scale = float(b.grad.abs().max()) + 1e-12
        assert float((a.grad - b.grad).abs().max()) / scale < 5e-4, name


def test_fused_shade_kernel_full_roughness_range_vs_fp64(golden_rotated):
    """Roughness over the model's whole range [0.09, 0.99] (primary.py: brdf[..., 3] * 0.9 + 0.09).  Below ~0.25 GGX's
    nom0 = NoH^2 (alpha^2 - 1) + 1 cancels catastrophically near the specular peak, so two fp32 evaluation orders differ
    by ~1e-3 and comparing them with each other says little; both are compared with the SAME expressions in fp64 instead:
    the kernel is at least as close to the exact value as the reference's fp32 torch evaluation (x2 + 1e-6 slack)."""
    from tensoir_b200.shade import shade
    f = oracle_field(golden_rotated)
    g = torch.Generator().manual_seed(9)
    bs, nl = 64, 512
    nrm = torch.nn.functional.normalize(torch.randn(bs, 3, generator=g), dim=-1)
    alb, fres = torch.rand(bs, 3, generator=g), torch.full((bs, 3), 0.04)
    rough = (torch.rand(bs, 1, generator=g) * 0.9 + 0.09).repeat(1, 3)
    rough[:8] = 0.09                                                     # the lower end explicitly
    view = torch.nn.functional.normalize(torch.randn(bs, 3, generator=g), dim=-1)
    direct = torch.rand(1, nl, 3, generator=g) * 2
    vis, ind = torch.rand(bs, nl, 1, generator=g), torch.rand(bs, nl, 3, generator=g) * 0.3
    li = torch.zeros(bs, 1, dtype=torch.long)
    torch.manual_seed(1)
    dirs = O.gen_light_incident_dirs(f, 'stratified_sampling')
    w = O.generate_envir_map_dir(16, 32)[0]

    def ref(dt):
        n_, a_, r_, f_, d_, v_, dr, ww, vs, ii = (t.to(DEV, dt) for t in (nrm, alb, rough, fres, direct, view, dirs, w,
                                                                         vis, ind))
        surf2l = dr[None].expand(bs, -1, -1)
        cos = torch.clamp(torch.einsum("ijk,ik->ij", surf2l, n_), min=0.0)
        brdf = a_.unsqueeze(1) / torch.pi + O.ggx_specular(n_, v_, surf2l, r_, f_)
        light = vs * d_[0][None] + ii
        return torch.sum(brdf * light * cos[:, :, None] * ww[None, :, None], dim=1)
    exact, ref32 = ref(torch.float64), ref(torch.float32)
    got = shade(*(t.to(DEV) for t in (nrm, alb, rough, fres, direct, view, li, dirs, w, vis, ind)))
    scale = exact.abs().clamp_min(1e-3)
    e_ours = float(((got.double() - exact).abs() / scale).max())
    e_ref = float(((ref32.double() - exact).abs() / scale).max())
    assert e_ours <= 2 * e_ref + 1e-6, (e_ours, e_ref)
    assert e_ours < 5e-3, e_ours


def test_relight_chunk(golden_rotated):
    """scripts/relight_importance.py chunk body through the fused density march, with the reference's recorded
    multinomial indices; plus one full relight_view with the inverse-CDF sampler (finite, in range, deterministic
    background)."""
    from tensoir_b200.relight import Environment_Light, relight_chunk, relight_view
    fx = golden_rotated
    m = model_from_fixture(fx, DEV)
    env = Environment_Light({"sunny": fx["env_rgb"].numpy()}, device=DEV)
    maps = tuple(t.to(DEV) for t in fx["relight_maps"])
    w, wo = relight_chunk(m, env, "sunny", fx["rays"].to(DEV), maps, 1.7, fx["relight_idx"].to(DEV), 64)
    close(wo, fx["relight_without_bg"], TOL, "relight without bg")
    close(w, fx["relight_with_bg"], TOL, "relight with bg")
    torch.manual_seed(3)
    res = relight_view(m, env, ["sunny"], fx["rays"].to(DEV), batch_size=40, num_samples=128)
    wv, wov = res["sunny"]
    assert wv.shape == (64, 3) and torch.isfinite(wv).all() and float(wv.min()) >= 0 and float(wv.max()) <= 1
    miss = res["_primary"][5] <= 0.5
    assert torch.equal(wov[miss], torch.ones_like(wov[miss]))


def test_config3_128_secondary_directions(golden_rotated):
    """BASELINE config 3 variant: an 8x16 = 128-direction environment grid (constructor kwargs envmap_h / envmap_w,
    tensorBase_rotated_lights.py:362-363) through the whole boundary, vs the oracle with the same grid."""
    from tensoir_b200 import Renderer_TensoIR_train, TensorVMSplit, AlphaGridMask
    fx = golden_rotated
    m = TensorVMSplit(fx["aabb"].to(DEV), fx["grid_size"], DEV, density_n_comp=[16] * 3, appearance_n_comp=[48] * 3,
                      app_dim=27, near_far=[2.0, 6.0], shadingMode='MLP_Fea', step_ratio=0.5, pos_pe=2, view_pe=2,
                      fea_pe=2, featureC=128, normals_kind='derived_plus_predicted', light_rotation=['000', '120'],
                      light_kind='sg', numLgtSGs=128, envmap_h=8, envmap_w=16)
    m.load_state_dict({k: v.to(DEV) for k, v in fx["state_dict"].items()})
    m.alphaMask = AlphaGridMask(DEV, fx["alpha_aabb"].to(DEV), fx["alpha_volume"].to(DEV))
    f = oracle_field(fx)
    f.envmap_h, f.envmap_w = 8, 16
    m.__dict__["_tir_randn_like"] = lambda t: torch.randn(t.shape).to(t.device)
    for method in ('fixed_envirmap', 'stratified_sampling'):
        torch.manual_seed(13)
        with torch.no_grad():
            got = Renderer_TensoIR_train(fx["rays"], None, fx["light_idx"], m, N_samples=-1, is_train=False,
                                         is_relight=True, sample_method=method, device=DEV, args=renderer_args(32))
        torch.manual_seed(13)
        want = O.renderer_train(f, fx["rays"], fx["light_idx"], -1, True, False, True, method, 160000, 32)
        for k in ("rgb_with_brdf_map", "rgb_map", "normal_map", "acc_map"):
            close(got[k], want[k], TOL, f"{method}:{k}")


def test_lean_counter_mode_is_bit_identical(rot):
    """TIR_MARCH_LEAN_COUNTERS (production mode): skipping the rest of a ray whose transmittance is exactly 0 changes no
    output beyond summation-order noise, no appearance sample and no ray count; only the mask / density counters shrink."""
    from tensoir_b200 import ops
    fx, m = rot
    pts, dirs, li = fx["surf"].to(DEV), fx["dirs"].to(DEV), fx["li2"].to(DEV)
    table = ops.equal_z_table(96, 0.05, 1.5, DEV)
    res = []
    for lean in (False, True):
        m.__dict__["_tir_lean"] = lean
        cnt = ops.new_counters(DEV)
        t, a, d, rgb, sc = ops.march_radiance(m, pts, dirs, li, table=table, counters=cnt)
        lst = sc.samples()
        order = torch.argsort(lst["ray"].long() * 4096 + lst["sample"].long())
        res.append((t, a, d, rgb, {k: v[order] for k, v in lst.items()}, ops.counters_dict(cnt)))
    m.__dict__.pop("_tir_lean")
    (t0, a0, d0, r0, l0, c0), (t1, a1, d1, r1, l1, c1) = res
    # skipped samples carry weight exactly 0; what may move is the association of the warp scans (the gather batches are
    # composed differently), i.e. the last bit
    close(t0, t1, 1e-6, "t_last"), close(a0, a1, 1e-6, "acc"), close(d0, d1, 1e-6, "depth"), close(r0, r1, 1e-6, "rgb")
    for k in ("ray", "sample"):
        assert torch.equal(l0[k], l1[k]), k         # the appearance list is the same set of samples
    close(l0["weight"], l1["weight"], 1e-6, "weight")
    assert c0["rays"] == c1["rays"] and c0["app"] == c1["app"]
    assert c1["mask"] <= c0["mask"] and c1["density"] <= c0["density"]


def _torch_tail(w, ray, rgb, brdf, brdfj, vn, dn, viewdirs, n_rays, model):
    """The torch expressions the fused tail replaces (tensorBase_rotated_lights.py:930-975)."""
    v_alb, v_rough = brdf[..., :3], brdf[..., 3:4] * 0.9 + 0.09
    a_cost = model.compute_relative_smoothness_loss(v_alb, brdfj[..., :3])
    r_cost = model.compute_relative_smoothness_loss(v_rough, brdfj[..., 3:4] * 0.9 + 0.09)
    vd = viewdirs.index_select(0, ray)
    if dn is not None:
        nd = torch.sum(torch.pow(vn - dn, 2), dim=-1, keepdim=True)
        no = torch.sum(vd * vn, dim=-1, keepdim=True).clamp(min=0)
    else:
        nd = no = torch.zeros_like(a_cost)
    vals = torch.cat([rgb, vn, v_alb, v_rough, a_cost, r_cost, nd, no], dim=-1)
    return torch.zeros(n_rays, 14, device=w.device).index_add_(0, ray, w[:, None] * vals)


def _torch_epilogue(packed, acc, depth, rays, fresnel0, bg):
    """The per-ray end of TensorBase.forward in torch (tensorBase_rotated_lights.py:977-1036)."""
    from tensoir_b200.relight_utils import linear2srgb_torch
    rgb, normal, albedo = packed[:, 0:3], packed[:, 3:6], packed[:, 6:9]
    rough, ac, rc, nd, no = packed[:, 9:10], packed[:, 10:11], packed[:, 11:12], packed[:, 12:13], packed[:, 13:14]
    fres = torch.zeros_like(albedo).fill_(fresnel0)
    if bg:
        depth = depth + (1. - acc) * rays[..., -1]
        rgb = rgb + (1. - acc[..., None])
        normal = normal + (1 - acc[..., None]) * torch.tensor([0., 0., 1.], device=packed.device)
        albedo, rough, fres = albedo + (1 - acc[..., None]), rough + (1 - acc[..., None]), fres + (1 - acc[..., None])
    return (linear2srgb_torch(rgb.clamp(0, 1)), depth, torch.nn.functional.normalize(normal, p=2, dim=-1, eps=1e-6),
            albedo.clamp(0, 1), rough.clamp(0, 1), fres.clamp(0, 1), nd, no, acc > 0.5, ac.mean(), rc.mean())


@pytest.mark.parametrize("both", [True, False])
def test_fused_tail_kernel_vs_autograd(rot, both):
    from tensoir_b200 import tail
    _, m = rot
    torch.manual_seed(3)
    n, n_rays = 5000, 512
    ray = torch.sort(torch.randint(0, n_rays, (n,), device=DEV))[0]
    w = torch.rand(n, device=DEV) * 0.3
    w[::17] = 0.0                                                        # padding rows of a static-capacity list
    rgb, brdf, brdfj = torch.rand(n, 3, device=DEV), torch.rand(n, 4, device=DEV), torch.rand(n, 4, device=DEV)
    vn = torch.nn.functional.normalize(torch.randn(n, 3, device=DEV), dim=-1)
    dn = torch.nn.functional.normalize(torch.randn(n, 3, device=DEV), dim=-1) if both else None
    vd = torch.nn.functional.normalize(torch.randn(n_rays, 3, device=DEV), dim=-1)
    G = torch.randn(n_rays, 14, device=DEV)
    res = []
    for fn in (lambda *a: tail.fused_tail(*a), lambda *a: _torch_tail(*a, m)):
        leaves = [t.clone().requires_grad_(True) for t in (w, rgb, brdf, brdfj, vn)] + \
                 ([dn.clone().requires_grad_(True)] if both else [])
        out = fn(leaves[0], ray, leaves[1], leaves[2], leaves[3], leaves[4], leaves[5] if both else None, vd, n_rays)
        out.backward(G)
        res.append([out.detach()] + [l.grad for l in leaves])
    for k, (g, wnt) in enumerate(zip(*res)):
        close(g, wnt, 2e-4, f"tail[{k}]")


@pytest.mark.parametrize("bg", [True, False])
def test_fused_epilogue_kernel_vs_autograd(rot, bg):
    from tensoir_b200 import tail
    torch.manual_seed(9)
    n = 2048
    packed = torch.rand(n, 14, device=DEV) * 1.3 - 0.1                    # some channels outside [0,1]: clamp gates
    packed[:100, 0:3] *= 0.002                                           # linear branch of the sRGB curve
    acc = torch.rand(n, device=DEV)
    acc[100:200] = 1.0
    depth, rays = torch.rand(n, device=DEV) * 4, torch.randn(n, 6, device=DEV)
    gs = None
    res = []
    for fn in (tail.epilogue, _torch_epilogue):
        leaves = [t.clone().requires_grad_(True) for t in (packed, acc, depth)]
        outs = fn(leaves[0], leaves[1], leaves[2], rays, 0.04, bg)
        # the fresnel map is a constant when no background is composited: no gradient to compare
        diff = [o for k, o in enumerate(outs) if o.dtype != torch.bool and (bg or k != 5)]
        if gs is None:
            gs = [torch.randn_like(o) for o in diff]
        torch.autograd.backward(diff, gs)
        res.append((outs, [l.grad if l.grad is not None else torch.zeros_like(l) for l in leaves]))
    for k, (g, wnt) in enumerate(zip(res[0][0], res[1][0])):
        if g.dtype == torch.bool:
            assert torch.equal(g, wnt)
        else:
            close(g, wnt.reshape(g.shape), 1e-4, f"epilogue out[{k}]")
    for k, (g, wnt) in enumerate(zip(res[0][1], res[1][1])):
        close(g, wnt, 2e-3, f"epilogue grad[{k}]")


@pytest.mark.parametrize("kind", ["derived_plus_predicted", "purely_predicted", "purely_derived"])
def test_fused_primary_matches_modular_path(golden_rotated, kind):
    """The fused primary march (tir_primary_march / _app_list / _heads / _backward: 21 launches, own backward kernels for
    the heads) against the modular autograd path (one kernel per op, torch / cuBLAS backward of the heads): every map and
    every parameter gradient, for the three normals kinds."""
    from tensoir_b200 import Renderer_TensoIR_train
    fx = golden_rotated
    rays, li = fx["rays"].to(DEV), fx["light_idx"].to(DEV)
    outs = []
    for modular in (True, False):
        m = model_from_fixture(fx, DEV)
        m.normals_kind = kind
        m.__dict__["_tir_modular"] = modular
        m.__dict__["_tir_randn_like"] = lambda t: torch.sin(t * 977.0)
        torch.manual_seed(11)
        got = Renderer_TensoIR_train(rays, None, li, m, N_samples=60, white_bg=True, is_train=True, is_relight=True,
                                     sample_method='stratified_sampling', device=DEV, args=renderer_args(24))
        loss = _train_loss(got) + 0.3 * got["acc_map"].mean() + 0.1 * got["depth_map"].mean() \
            + 0.05 * (got["albedo_map"] ** 2).mean() + 0.05 * (got["roughness_map"] ** 2).mean() \
            + 0.05 * (got["normal_map"][:, 2]).mean()
        loss.backward()
        outs.append((got, loss, {k: p.grad.detach().clone() for k, p in m.named_parameters() if p.grad is not None}))
    (g0, l0, gr0), (g1, l1, gr1) = outs
    for k in g0:
        close(g1[k], g0[k], 2e-5, k)
    close(l1, l0, 2e-5, "loss")
    assert set(gr0) == set(gr1), set(gr0) ^ set(gr1)
    worst = {}
    for k in gr0:
        scale = float(gr0[k].abs().max()) + 1e-12
        worst[k] = float((gr0[k] - gr1[k]).abs().max()) / scale
    bad = {k: v for k, v in worst.items() if v > 2e-4}
    assert not bad, bad


def test_tcgen05_mlp_matches_mma_sync_kernel(rot):
    """The sm_100a-native appearance MLP (tcgen05.mma, accumulator + activations in TMEM, csrc/tir_mlp_tc5.cu) against
    the round-1 mma.sync kernel: explicit points for the three heads (ragged sizes incl. a partial tile and an odd
    number of tiles), and the secondary appearance list; no bounded wait may have timed out."""
    import ctypes as C
    from tensoir_b200 import _lib, ops
    from tensoir_b200.device_field import mlp_struct
    fx, m = rot
    lib = _lib.load()
    f = ops.device_field(m).refresh(m)
    g = torch.Generator().manual_seed(7)
    for n in (1, 127, 128, 300, 5000):
        xn = (torch.rand(n, 3, generator=g) * 1.9 - 0.95).to(DEV)
        xi = torch.nn.functional.normalize(torch.randn(n, 3, generator=g), dim=-1).to(DEV)
        li = torch.zeros(n, dtype=torch.int32, device=DEV)
        for head, light, act in (("renderModule", "index", 0), ("renderModule_brdf", "mean", 0),
                                 ("renderModule_normal", "mean", 1)):
            keep = []
            mlp = mlp_struct(m, head, keep, light=light)
            outs = []
            for fn in (lib.tir_app_mlp_points_legacy, lib.tir_app_mlp_points_tc5):
                out = torch.full((n, mlp.out_dim), -7.0, device=DEV)
                _lib.check(fn(C.byref(f), C.byref(mlp), _lib.dptr(xn), _lib.dptr(xi),
                              _lib.dptr(li, torch.int32) if light == "index" else None, n, act, _lib.dptr(out),
                              _lib.stream_ptr()), "mlp points")
                outs.append(out)
            torch.cuda.synchronize()
            assert lib.tir_mlp_tc5_error() == 0
            close(outs[1], outs[0], 2e-5, f"{head} n={n}")
    # sample-list form on a real secondary march
    with torch.no_grad():
        out = m(fx["rays"].to(DEV), fx["light_idx"].to(DEV), is_train=False, is_relight=True, N_samples=-1)
    rays = fx["rays"].to(DEV)
    mask = out[9]
    surf = (rays[:, :3] + out[1][:, None] * rays[:, 3:])[mask]
    dirs = m.gen_light_incident_dirs(method='fixed_envirmap').to(DEV)
    st = ops.SecondaryStages(m, surf, out[2][mask], fx["light_idx"].to(DEV)[mask], dirs, n_sample=24)
    st.march()
    res = []
    for fn in (lib.tir_app_mlp_legacy, lib.tir_app_mlp_tc5):
        st.ind.zero_()
        _lib.check(fn(C.byref(st.f), C.byref(st.mlp_s), _lib.dptr(st.sc.buf, torch.uint8),
                      _lib.dptr(st.sc.count, torch.int32), st.sc.capacity, _lib.dptr(st.dr), st.n_dirs,
                      _lib.dptr(st.li, torch.int32), _lib.dptr(st.ind), _lib.stream_ptr()), "mlp list")
        res.append(st.ind.clone())
    torch.cuda.synchronize()
    assert lib.tir_mlp_tc5_error() == 0
    assert int(st.sc.count.item()) > 100
    close(res[1], res[0], 2e-5, "indirect light")


def _lego_pair(grid):
    """(CUDA model, oracle field) of the bench scene at ``grid``^3: same seed, same init order (bench.make_lego_state)."""
    import bench
    from tensoir_b200.synthetic import make_lego_model
    import contextlib
    import io
    with contextlib.redirect_stdout(io.StringIO()):
        model = make_lego_model(grid, DEV)
    return model, bench.make_lego_state(grid)


def test_baseline_shape_vs_oracle():
    """The BASELINE workload shape (lego-shaped scene, 4096-ray training batch of the 800x800 views, N_samples =
    n_samples_for(grid), 16x32 secondary directions x 96 samples), not a toy fixture: the CUDA boundary against the
    oracle on a 256-ray subsample of the same batch — mask / density / appearance / ray COUNTS exact, every map 1e-4."""
    import bench
    from tensoir_b200 import Renderer_TensoIR_train, ops
    from tensoir_b200.synthetic import hemisphere_poses, training_batch, n_samples_for
    grid = 128
    model, field = _lego_pair(grid)
    n_s = n_samples_for(grid)
    rays, li = training_batch(hemisphere_poses(100), 4096, 3)
    sub = torch.arange(0, 4096, 16)                       # 256 rays spread over the batch
    r_s, l_s = rays[sub].contiguous(), li[sub].contiguous()
    counters = ops.new_counters(DEV)
    with torch.no_grad():
        full = Renderer_TensoIR_train(rays, None, li, model, N_samples=n_s, white_bg=True, is_train=False,
                                      is_relight=True, sample_method='fixed_envirmap', device=DEV, args=bench.Args)
        model.__dict__["_tir_counters"] = counters
        part = Renderer_TensoIR_train(r_s, None, l_s, model, N_samples=n_s, white_bg=True, is_train=False,
                                      is_relight=True, sample_method='fixed_envirmap', device=DEV, args=bench.Args)
        model.__dict__.pop("_tir_counters")
        field.counters.clear()
        want = O.renderer_train(field, r_s, l_s, n_s, True, False, True, 'fixed_envirmap', 160000, 96, 0.05, 1.5)
    got_c = ops.counters_dict(counters)
    assert got_c["overflow"] == 0
    hits = int(want["acc_map"].gt(0.5).sum())
    assert hits > 40, hits                                 # the subsample really exercises the secondary path
    for k in ("rgb_map", "depth_map", "normal_map", "albedo_map", "roughness_map", "acc_map", "rgb_with_brdf_map",
              "normals_orientation_loss_map"):
        close(part[k], want[k], TOL, k)
        close(full[k][sub.to(DEV)], want[k], TOL, "full batch " + k)     # rays are independent of their batch
    # normals_diff_map = sum_s w |n_pred - n_derived|^2 with n_derived = -normalize(d sigma / d x).  Inside the solid boxes
    # of this scene the density planes are 30 + 1e-3 noise, so the spatial derivative is a DIFFERENCE of tap sums of size
    # ~30 whose result is ~1e-3: cancellation leaves ~2e-3 relative error that depends on the summation order (the
    # reference's own CPU and CUDA runs differ the same way).  Most rays still agree to 1e-4; every ray within 2 %.
    err = (part["normals_diff_map"].cpu() - want["normals_diff_map"]).abs()
    ok = err <= TOL * (1 + want["normals_diff_map"].abs())
    assert float(ok.float().mean()) > 0.8, float(ok.float().mean())
    assert float(err.max()) < 0.02 * float(want["normals_diff_map"].abs().max().clamp_min(1.0)), float(err.max())
    oc = field.counters
    assert got_c["rays"] == 256 + oc["secondary_rays"], (got_c, dict(oc))
    # the oracle counts one appearance gather per compute_*feature CALL: the primary samples are visited twice (at the
    # sample points and at the jittered points, tensorBase:930-940), the CUDA counter counts appearance SAMPLES
    c1 = ops.new_counters(DEV)
    model.__dict__["_tir_counters"] = c1
    with torch.no_grad():
        model(r_s.to(DEV), l_s.to(DEV), is_train=False, is_relight=True, N_samples=n_s)
    model.__dict__.pop("_tir_counters")
    n_app_primary = ops.counters_dict(c1)["app"]
    assert got_c["mask"] == oc["mask"], (got_c, dict(oc))
    assert got_c["app"] + n_app_primary == oc["app"], (got_c, n_app_primary, dict(oc))
    # valid density samples: exact on every golden fixture; at this size (1.04 M samples) ONE sample differs - the
    # alpha-mask test `trilinear(binary volume) > 0` is evaluated exactly here (some corner with positive weights is
    # set), while the float product of three weights can underflow to 0 in the reference
    assert abs(got_c["density"] - oc["density"]) <= 2, (got_c, dict(oc))
    assert psnr(part["rgb_with_brdf_map"], want["rgb_with_brdf_map"]) > 60


def test_graph_replay_tracks_eager_training_for_50_steps():
    """50 consecutive training steps of the bench scene (128^3, 1024-ray batches, Adam): CUDA-graph replay (static
    lists, device-side counts) against the eager step on identical batches and identical host randoms.  Losses agree
    step by step and the parameters end up together (atomics order is the only difference); no replay overflowed."""
    import bench
    from tensoir_b200 import Renderer_TensoIR_train
    from tensoir_b200.static_step import StaticTrainStep
    from tensoir_b200.synthetic import hemisphere_poses, training_batch, n_samples_for
    grid, n_rays, steps = 128, 1024, 50
    n_s = n_samples_for(grid)
    poses = hemisphere_poses(100)
    batches = [tuple(t.to(DEV) for t in training_batch(poses, n_rays, it)) for it in range(steps)]
    target = torch.full((n_rays, 3), 0.5, device=DEV)
    g = torch.Generator().manual_seed(5)
    jit = [torch.rand(n_rays, 1, generator=g) for _ in range(steps)]
    runs = []
    for graphed in (False, True):
        model, _ = _lego_pair(grid)
        model.__dict__["_tir_randn_like"] = lambda t: torch.sin(t * 977.0)
        fixed_dirs = model.gen_light_incident_dirs(method='fixed_envirmap').to(DEV)
        opt = torch.optim.Adam(model.get_optparam_groups(0.02, 0.001), betas=(0.9, 0.99), fused=True,
                               capturable=graphed)
        losses = []
        if graphed:
            st = StaticTrainStep(model, opt, n_rays, n_s, bench.Args, lambda ret, m: bench.loss_of(ret, target, m),
                                 sample_method='fixed_envirmap', device=DEV, lag=1)
            st.calibrate(batches[:4])
            it_box = [0]

            def stage(slot, st=st):
                st.static["jitter"].copy_(jit[min(it_box[0], steps - 1)])
                st.static["dirs"].copy_(fixed_dirs)
            st._stage_host_randoms = stage
            st.capture(warmup=1)
            for it, (rays, li) in enumerate(batches):
                it_box[0] = it
                losses.append(st.run(rays, li).detach().clone())
            st.flush()
            assert st.overflowed() == 0 and st.redone == 0
            st.release()
        else:
            for it, (rays, li) in enumerate(batches):
                torch.manual_seed(1000 + it)
                torch.rand = _FixedRand(jit[it])           # the per-ray jitter the graph run stages for this step
                try:
                    ret = Renderer_TensoIR_train(rays, None, li, model, N_samples=n_s, white_bg=True, is_train=True,
                                                 is_relight=True, sample_method='fixed_envirmap', device=DEV,
                                                 args=bench.Args)
                finally:
                    torch.rand = _FixedRand.orig
                loss = bench.loss_of(ret, target, model)
                opt.zero_grad(set_to_none=True)
                loss.backward()
                opt.step()
                losses.append(loss.detach().clone())
        runs.append((torch.stack(losses).cpu(), {k: p.detach().clone() for k, p in model.named_parameters()}))
    (l0, p0), (l1, p1) = runs
    assert torch.isfinite(l0).all() and torch.isfinite(l1).all()
    assert float(l0[-1]) < float(l0[0])                                  # it trains
    rel = ((l0 - l1).abs() / l0.abs().clamp_min(1e-6)).max()
    assert float(rel) < 2e-3, float(rel)
    for k in p0:
        d = float((p0[k] - p1[k]).abs().max())
        # Adam divides by sqrt(v): entries whose gradients are atomics-order noise wander by up to ~lr per step, so after
        # 50 steps the parameters agree to a few percent of their range while the loss curves agree to 2e-3
        assert d <= 5e-2 * max(float(p0[k].abs().max()), 1e-2), (k, d)


class _FixedRand:
    """torch.rand stand-in for one eager step: the first [n,1] request returns the staged per-ray jitter."""
    orig = torch.rand

    def __init__(self, value):
        self.value, self.used = value, False

    def __call__(self, *size, **kw):
        shape = tuple(size[0]) if len(size) == 1 and isinstance(size[0], (tuple, list, torch.Size)) else tuple(size)
        if not self.used and shape == tuple(self.value.shape):
            self.used = True
            return self.value.clone()
        return _FixedRand.orig(*size, **kw)


def test_fused_adam_matches_torch_adam():
    """tensoir_b200.optim.FusedAdam against torch.optim.Adam over 6 steps: plain, channel-last and odd-sized tensors,
    two learning rates, the L1 term against autograd of w * |x|.sum(), gradients cleared in place, and the found_inf skip
    (parameters, moments and step counter untouched)."""
    from tensoir_b200.optim import FusedAdam
    g = torch.Generator().manual_seed(3)
    shapes = [(1, 16, 33, 29), (1, 48, 17, 1), (128, 150), (7,), (4099,)]
    def make():
        ps = []
        for i, sh in enumerate(shapes):
            t = torch.randn(sh, generator=g).to(DEV)
            if len(sh) == 4:
                t = t.contiguous(memory_format=torch.channels_last)
            ps.append(torch.nn.Parameter(t))
        return ps
    g.manual_seed(3); pa = make()
    g.manual_seed(3); pb = make()
    l1w = 3e-3
    oa = torch.optim.Adam([{"params": pa[:2], "lr": 0.02}, {"params": pa[2:], "lr": 1e-3}], betas=(0.9, 0.99))
    ob = FusedAdam([{"params": pb[:2], "lr": 0.02}, {"params": pb[2:], "lr": 1e-3}], betas=(0.9, 0.99),
                   l1={pb[0]: l1w})
    flag = torch.zeros((), device=DEV)
    ob.found_inf = flag
    for it in range(6):
        gs = [torch.randn(p.shape, generator=g).to(DEV) for p in pa]
        for p, q, gr in zip(pa, pb, gs):
            gr = gr.contiguous(memory_format=torch.channels_last) if gr.dim() == 4 else gr
            p.grad = gr.clone() + (l1w * torch.sign(p.detach()) if p is pa[0] else 0)
            if q.grad is None:
                q.grad = gr.clone()
            else:
                assert float(q.grad.abs().max()) == 0.0            # cleared in place by the previous step
                q.grad.add_(gr)
        if it == 3:                                                # a skipped step: nothing but the gradients changes
            flag.fill_(1.0)
            before = [q.detach().clone() for q in pb]
            ob.step()
            flag.zero_()
            assert all(torch.equal(x, q.detach()) for x, q in zip(before, pb))
            for q, gr in zip(pb, gs):
                q.grad.add_(gr.contiguous(memory_format=torch.channels_last) if gr.dim() == 4 else gr)
        oa.step()
        ob.step()
    for p, q in zip(pa, pb):
        assert float((p - q).abs().max()) < 2e-6 * max(1.0, float(p.abs().max())), float((p - q).abs().max())
    assert float(ob.state[pb[0]]["step"]) == 6.0


def test_device_ray_generation_matches_host_rays():
    """tir_generate_rays (rays of (view, pixel) ids on the device) against the host construction the datasets use
    (get_ray_directions + normalise + get_rays, restated in tensoir_b200.synthetic.pixel_rays)."""
    from tensoir_b200 import ops
    from tensoir_b200.synthetic import hemisphere_poses, pixel_rays
    poses = hemisphere_poses(100)
    g = torch.Generator().manual_seed(1)
    view = torch.randint(0, 100, (5000,), generator=g, dtype=torch.int32)
    pix = torch.randint(0, 800 * 800, (5000,), generator=g, dtype=torch.int32)
    want = torch.empty(5000, 6)
    for v in view.unique().tolist():
        m = view == v
        want[m] = pixel_rays(poses[v], pix[m].long())
    got = ops.generate_rays(poses.to(DEV), view.to(DEV), pix.to(DEV)).cpu()
    assert torch.equal(got[:, :3], want[:, :3])
    assert float((got[:, 3:] - want[:, 3:]).abs().max()) < 3e-7
    assert float((got[:, 3:].norm(dim=-1) - 1).abs().max()) < 1e-6


class _TVLoss(torch.nn.Module):
    """utils.TVLoss (utils.py:143-162), restated for the test."""

    def __init__(self, TVLoss_weight=1):
        super().__init__()
        self.TVLoss_weight = TVLoss_weight

    def forward(self, x):
        b, _, h, w = x.shape
        ch, cw = x[:, :, 1:, :].numel() // b, x[:, :, :, 1:].numel() // b
        return self.TVLoss_weight * 2 * (torch.pow(x[:, :, 1:, :] - x[:, :, :h - 1, :], 2).sum() / ch
                                         + torch.pow(x[:, :, :, 1:] - x[:, :, :, :w - 1], 2).sum() / cw) / b


def test_fused_tv_matches_torch_autograd(golden_rotated):
    """tv.tv_planes (one forward + one backward launch for the three planes) against autograd of the reference's TVLoss
    expression: channel-last parameters (16 / 48 / 6 channels -> vector and scalar kernels), plain NCHW tensors, a decayed
    loss weight, gradients handed to autograd and accumulated in place into an existing .grad."""
    from tensoir_b200 import tv, _lib
    g = torch.Generator().manual_seed(11)
    reg = _TVLoss(1.7)

    def planes(shapes, channel_last):
        out = []
        for sh in shapes:
            t = torch.randn(sh, generator=g).to(DEV)
            if channel_last:
                t = t.contiguous(memory_format=torch.channels_last)
            out.append(torch.nn.Parameter(t))
        return out
    cases = [([(1, 16, 37, 29), (1, 16, 29, 41), (1, 16, 41, 37)], True),
             ([(1, 48, 21, 19), (1, 48, 19, 23), (1, 48, 23, 21)], True),
             ([(1, 6, 9, 7), (1, 6, 7, 5)], True),
             ([(1, 16, 13, 11), (1, 5, 8, 9), (1, 4, 6, 7)], False)]
    for shapes, cl in cases:
        ps = planes(shapes, cl)
        qs = [torch.nn.Parameter(p.detach().clone(memory_format=torch.preserve_format)) for p in ps]
        w = 0.05 * 0.9993
        before = _lib.launch_count
        ours = tv.tv_planes(ps, reg, 1e-2, inplace=False) * w
        assert _lib.launch_count - before == 1
        ref = sum(reg(q) * 1e-2 for q in qs) * w
        assert abs(float(ours) - float(ref)) < 1e-5 * abs(float(ref)), (float(ours), float(ref))
        ours.backward()
        ref.backward()
        assert _lib.launch_count - before == 2
        for p, q in zip(ps, qs):
            scale = float(q.grad.abs().max())
            assert float((p.grad - q.grad).abs().max()) < 1e-5 * scale, (shapes, cl)
        # second pass: .grad exists -> accumulated in place (no buffer handed to autograd), twice the gradient
        held = [p.grad for p in ps]
        (tv.tv_planes(ps, reg, 1e-2, inplace=True) * w).backward()
        for p, q, h in zip(ps, qs, held):
            assert p.grad is h
            assert float((p.grad - 2 * q.grad).abs().max()) < 2e-5 * float(q.grad.abs().max())
    # the model methods route through it (density: 3 planes in one launch) and keep the reference's values
    m = model_from_fixture(golden_rotated, DEV)
    before = _lib.launch_count
    val = m.TV_loss_density(reg) + m.TV_loss_app(reg)
    assert _lib.launch_count - before == 2
    want = sum(reg(p) * 1e-2 for p in m.density_plane) + sum(reg(p) * 1e-2 for p in m.app_plane)
    assert abs(float(val) - float(want)) < 1e-5 * abs(float(want))
    # a callable that is not the reference's TVLoss is simply called
    assert torch.allclose(m.TV_loss_density(lambda x: x.abs().mean()), sum(p.abs().mean() * 1e-2 for p in m.density_plane))
