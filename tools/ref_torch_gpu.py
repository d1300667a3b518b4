"""PyTorch-on-B200 denominator: the UNMODIFIED reference modules (bench.py --reference: models.tensoRF_rotated_lights +
renderer.Renderer_TensoIR_train, eager PyTorch, no tensoir_b200 code on the path) timed on the same GPU, the same
field (loaded from a checkpoint bench.py wrote in the reference's format) and the same ray batches as bench.py.
Run by bench.py in a subprocess, from the reference's directory:
    PYTHONPATH=tools/ref_stubs:<reference>:<repo>  python -P tools/ref_torch_gpu.py ..."""
import argparse
import json
import os
import sys
import time

import torch

ap = argparse.ArgumentParser()
ap.add_argument("--ckpt", required=True)
ap.add_argument("--grid", type=int, default=300)
ap.add_argument("--batch", type=int, default=4096)
ap.add_argument("--steps", type=int, default=3)
ap.add_argument("--warmup", type=int, default=2)
ap.add_argument("--n_lights", type=int, default=1)
a = ap.parse_args()

from models.tensoRF_rotated_lights import TensorVMSplit, AlphaGridMask   # noqa: E402,F401  (the reference's own)
from renderer import Renderer_TensoIR_train                               # noqa: E402
import models.tensoRF_rotated_lights as _m                                # noqa: E402
assert os.path.abspath(_m.__file__).startswith(os.getcwd() + os.sep), _m.__file__     # not dropin/'s

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.append(ROOT)
from tensoir_b200.synthetic import hemisphere_poses, training_batch, n_samples_for   # noqa: E402  (ray generator only)

dev = torch.device("cuda", 0)
ckpt = torch.load(a.ckpt, map_location=dev, weights_only=False)
kw = ckpt["kwargs"]
kw.update({"device": dev})
model = TensorVMSplit(**kw)
model.load(ckpt)


class Args:
    second_nSample, second_near, second_far = 96, 0.05, 1.5


opt = torch.optim.Adam(model.get_optparam_groups(0.02, 0.001), betas=(0.9, 0.99))
poses = hemisphere_poses(100)
n_s = n_samples_for(a.grid)
target = torch.full((a.batch, 3), 0.5, device=dev)
ts = []
for it in range(a.warmup + a.steps):
    rays, li = training_batch(poses, a.batch, it, n_lights=a.n_lights)
    rays, li = rays.to(dev), li.to(dev)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    ret = Renderer_TensoIR_train(rays, None, li, model, N_samples=n_s, white_bg=True, is_train=True, is_relight=True,
                                 sample_method='stratified_sampling', chunk_size=160000, device=dev, args=Args)
    loss = torch.mean((ret['rgb_map'] - target) ** 2) + 4e-5 * model.density_L1()
    loss = loss + 0.2 * torch.mean((ret['rgb_with_brdf_map'] - target) ** 2)
    loss = loss + 0.0005 * ret['normals_diff_map'].mean() + 0.001 * ret['normals_orientation_loss_map'].mean()
    loss = loss + 0.001 * ret['roughness_smoothness_loss'] + 0.001 * ret['albedo_smoothness_loss']
    opt.zero_grad()
    loss.backward()
    opt.step()
    torch.cuda.synchronize()
    if it >= a.warmup:
        ts.append(time.perf_counter() - t0)
print(json.dumps({"impl": "unmodified reference modules, eager PyTorch, same B200 / field / batches",
                  "ms_per_step": 1e3 * sum(ts) / len(ts), "steps": a.steps, "warmup": a.warmup, "loss": float(loss),
                  "peak_mem_GB": torch.cuda.max_memory_allocated() / 1e9}))
