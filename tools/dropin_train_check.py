"""Drop-in check on a GPU: the UNMODIFIED reference script `train_tensoIR.py` (of the checkout given by --reference) is run
twice for a few iterations on a small synthetic on-disk dataset in the reference's own format —
  A. with `dropin/` first on PYTHONPATH: `models.*` / `renderer` resolve to tensoir_b200 (CUDA kernels),
  B. against the reference's own modules (eager PyTorch on the same GPU) —
same seeds, same config, and the per-iteration training losses written by the script's own SummaryWriter are compared.
The run crosses the script's `update_AlphaMask_list[0]` iteration, so both phases (radiance-only, then relight with
secondary rays), `filtering_rays`, `updateAlphaMask`, `shrink` and `save` are exercised through the drop-in surface.

    python tools/dropin_train_check.py --reference <original project> [--iters 24] [--out profiles/r2_dropin_train_check.json]
"""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = None           # the original project's checkout (--reference)
STUBS = os.path.join(ROOT, "tools", "ref_stubs")


def make_dataset(root, n_train=3, n_test=1):
    """TensoIR-synthetic layout (dataLoader/tensoIR_rotation_setting.py:86-140): <scan>/<split>_<id>/metadata.json +
    rgba_<light>_<rotation>.png, 800x800 RGBA."""
    from PIL import Image
    scan = os.path.join(root, "data", "lego")
    hdr = os.path.join(root, "hdr")
    os.makedirs(hdr, exist_ok=True)
    yy, xx = np.mgrid[0:800, 0:800].astype(np.float32)
    for split, n in (("train", n_train), ("test", n_test)):
        for i in range(n):
            d = os.path.join(scan, f"{split}_{i:03d}")
            os.makedirs(d, exist_ok=True)
            ang = 0.7 + 1.1 * i + (0.4 if split == "test" else 0.0)
            cam = np.array([4 * np.cos(ang) * 0.8, 4 * np.sin(ang) * 0.8, 2.4])
            fwd = -cam / np.linalg.norm(cam)
            right = np.cross(fwd, np.array([0, 0, 1.0])); right /= np.linalg.norm(right)
            up = np.cross(right, fwd)
            c2w = np.eye(4)
            c2w[:3, 0], c2w[:3, 1], c2w[:3, 2], c2w[:3, 3] = right, up, -fwd, cam       # blender convention
            meta = {"imw": 800, "imh": 800, "cam_angle_x": 0.6911112070083618,
                    "cam_transform_mat": ",".join(f"{v:.8f}" for v in c2w.reshape(-1))}
            json.dump(meta, open(os.path.join(d, "metadata.json"), "w"))
            r = np.sqrt((xx - 400 - 30 * i) ** 2 + (yy - 420) ** 2)
            alpha = (r < 230).astype(np.float32)
            rgb = np.stack([0.2 + 0.6 * xx / 800, 0.3 + 0.5 * yy / 800, 0.5 + 0.3 * np.cos(r / 60)], -1) * alpha[..., None]
            img = (np.concatenate([rgb, alpha[..., None]], -1) * 255).astype(np.uint8)
            Image.fromarray(img, "RGBA").save(os.path.join(d, "rgba_sunset_000.png"))
    return scan, hdr


def make_checkpoint(path):
    """Both arms start from the same checkpoint (the synthetic lego density field with the reference initialisation for
    everything else, written in the reference's checkpoint format by tensoir_b200's `save`): a few iterations from a
    random init leave the field empty, and the reference's own updateAlphaMask then fails on an empty mask."""
    code = ("import sys, torch; sys.path.insert(0, %r); import __graft_entry__ as g; g.build(); "
            "from tensoir_b200.synthetic import make_lego_model; m = make_lego_model(64, torch.device('cuda', 0)); "
            "m.alphaMask = None; m.save(%r)" % (ROOT, path))
    subprocess.run([sys.executable, "-c", code], check=True, stdout=subprocess.DEVNULL)


def write_config(path, scan, hdr, basedir, iters, ckpt):
    open(path, "w").write(f"""
ckpt = {ckpt}
dataset_name = tensoIR_unknown_rotated_lights
datadir = {scan}
hdrdir = {hdr}
expname = run
basedir = {basedir}
add_timestamp = 0
downsample_train = 8
downsample_test = 8
n_iters = {iters}
batch_size = 1024
lr_decay_iters = {iters}
N_voxel_init = 262144
N_voxel_final = 262144
upsamp_list = [100000000]
update_AlphaMask_list = [7, 100000000]
N_vis = 0
vis_every = 100000000
save_iters = 100000000
render_test = 0
progress_refresh_rate = 1
n_lamb_sigma = [16,16,16]
n_lamb_sh = [48,48,48]
model_name = TensorVMSplit
shadingMode = MLP_Fea
fea2denseAct = softplus
view_pe = 2
fea_pe = 2
pos_pe = 2
light_rotation = [000]
light_sample_train = stratified_sampling
light_kind = sg
numLgtSGs = 128
normals_kind = derived_plus_predicted
normals_diff_weight = 0.0005
normals_orientation_weight = 0.001
rgb_brdf_weight = 0.2
batch_size_test = 4096
light_name = sunset
albedo_smoothness_loss_weight = 0.001
roughness_smoothness_loss_weight = 0.001
L1_weight_inital = 8e-5
L1_weight_rest = 4e-5
rm_weight_mask_thre = 1e-4
TV_weight_density = 0.05
TV_weight_app = 0.005
""")


def scalars(logdir, tag):
    from tensorboard.backend.event_processing.event_accumulator import EventAccumulator
    acc = EventAccumulator(logdir, size_guidance={"scalars": 0})
    acc.Reload()
    return [(e.step, e.value) for e in acc.Scalars(tag)] if tag in acc.Tags()["scalars"] else []


def run(arm, cfg, env_paths, log):
    env = dict(os.environ)
    env["PYTHONPATH"] = os.pathsep.join(env_paths)
    env.pop("WORLD_SIZE", None)
    # -P: do not put the script's own directory first on sys.path - that directory holds the reference's models/ and
    # renderer.py, which would shadow dropin/ no matter what PYTHONPATH says (the script itself stays untouched)
    p = subprocess.run([sys.executable, "-P", "train_tensoIR.py", "--config", cfg], cwd=REF, env=env,
                       stdout=open(log, "w"), stderr=subprocess.STDOUT, timeout=1500)
    return p.returncode


def main():
    global REF
    ap = argparse.ArgumentParser()
    ap.add_argument("--reference", required=True, help="a checkout of the original TensoIR project")
    ap.add_argument("--iters", type=int, default=24)
    ap.add_argument("--out", default=None)
    ap.add_argument("--keep", action="store_true")
    a = ap.parse_args()
    REF = os.path.abspath(a.reference)
    if not os.path.isfile(os.path.join(REF, "train_tensoIR.py")):
        raise SystemExit(f"{REF}: not a checkout of the original project (no train_tensoIR.py)")
    tmp = tempfile.mkdtemp(prefix="tir_dropin_")
    scan, hdr = make_dataset(tmp)
    ckpt = os.path.join(tmp, "start.th")
    make_checkpoint(ckpt)
    res = {"what": "unmodified reference train_tensoIR.py, dropin/ (tensoir_b200 kernels) vs the reference's own modules "
                   "(eager PyTorch), same GPU, same seeds", "iters": a.iters}
    curves = {}
    for arm, paths in (("dropin", [STUBS, os.path.join(ROOT, "dropin"), ROOT, REF]), ("reference", [STUBS, REF])):
        base = os.path.join(tmp, "log_" + arm)
        cfg = os.path.join(tmp, f"cfg_{arm}.txt")
        write_config(cfg, scan, hdr, base, a.iters, ckpt)
        log = os.path.join(tmp, f"{arm}.log")
        rc = run(arm, cfg, paths, log)
        res[arm + "_rc"] = rc
        if rc != 0:
            res[arm + "_tail"] = open(log).read()[-3000:]
            continue
        logdir = os.path.join(base, "run")
        curves[arm] = {t: scalars(logdir, "train/" + t) for t in ("mse", "mse_rgb", "mse_rgb_brdf")}
        env = dict(os.environ, PYTHONPATH=os.pathsep.join(paths))
        who = subprocess.run([sys.executable, "-P", "-c", "import models.tensoRF_rotated_lights as m, renderer as r; "
                              "print(m.TensorVMSplit.__module__, r.Renderer_TensoIR_train.__module__)"], cwd=REF,
                             env=env, capture_output=True, text=True)
        res[arm + "_resolves_to"] = who.stdout.strip().splitlines()[-1] if who.stdout.strip() else who.stderr[-300:]
    if len(curves) == 2:
        for tag in ("mse", "mse_rgb", "mse_rgb_brdf"):
            x, y = curves["dropin"][tag], curves["reference"][tag]
            n = min(len(x), len(y))
            rel = [abs(x[i][1] - y[i][1]) / max(abs(y[i][1]), 1e-8) for i in range(n)]
            res[tag] = {"n": n, "dropin": [round(v[1], 6) for v in x[:n]], "reference": [round(v[1], 6) for v in y[:n]],
                        "max_rel_diff": max(rel) if rel else None}
        res["ok"] = bool(res["mse"]["n"] >= a.iters and res["mse"]["max_rel_diff"] < 0.05)
    else:
        res["ok"] = False
    out = json.dumps(res)
    print(out)
    if a.out:
        open(a.out, "w").write(out + "\n")
    if not a.keep:
        shutil.rmtree(tmp, ignore_errors=True)
    return 0 if res["ok"] else 1


if __name__ == "__main__":
    sys.exit(main())
