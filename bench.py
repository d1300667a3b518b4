#!/usr/bin/env python
"""bench.py — the driver's benchmark contract for tensoir_b200.

Step = one training step of the relight phase on one 4096-ray batch of the synthetic lego-shaped scene
(BASELINE.json configs[1]: single light, 800x800 x 100 train views, full VM grid + BRDF MLPs):
    Renderer_TensoIR_train(is_train=True, is_relight=True, stratified_sampling)   primary + secondary marches
    + loss assembly of train_tensoIR.py:262-312 + backward + Adam step.
Metric = (primary + secondary rays marched) / second, whole job.  `--impl reference` times the reference's
algorithm (the oracle port under oracle/, the only part of this file that may execute oracle/) on the host cores.
"""
import argparse
import contextlib
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True    # the benchmark writes nothing into the tree it runs from (it may be read-only)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import torch                      # noqa: E402
import torch.distributed as dist  # noqa: E402

METRIC = "primary+secondary rays/sec (800x800 lego-shaped synthetic, relight training step)"
UNIT = "rays/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--grid", type=int, default=300)
    ap.add_argument("--batch", type=int, default=4096)
    ap.add_argument("--cpu-rays", type=int, default=1024, help="bounded CPU-baseline sample (primary rays / step)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--eager", action="store_true", help="do not capture the step into a CUDA graph")
    ap.add_argument("--host-rays", dest="host_rays", action="store_true",
                    help="end-to-end arm: copy [n,6] rays from the host instead of generating them on the device from ids")
    ap.add_argument("--torch-adam", dest="torch_adam", action="store_true",
                    help="torch.optim.Adam(fused=True) + autograd density_L1 instead of tensoir_b200.optim.FusedAdam")
    ap.add_argument("--config", type=int, default=2, choices=[2, 3, 4, 5],
                    help="BASELINE.json configs index + 1: 2 single light (default, the metric's config), 3 rotated "
                         "multi-light with --envmap_h x --envmap_w secondary directions, 4 general multi-light, 5 relight pass")
    ap.add_argument("--envmap_h", type=int, default=None)
    ap.add_argument("--envmap_w", type=int, default=None)
    ap.add_argument("--no-strong", dest="no_strong", action="store_true",
                    help="N > 1: skip the additional strong-scaling measurement")
    ap.add_argument("--reference", default=None, metavar="DIR",
                    help="a checkout of the original TensoIR project: adds the PyTorch-on-GPU denominator (its unmodified "
                         "modules on the same GPU, field and batches)")
    ap.add_argument("--no-torch-reference", dest="no_torch_reference", action="store_true",
                    help="skip the PyTorch-on-GPU denominator even with --reference")
    ap.add_argument("--dump-outputs", dest="dump_outputs", default=None, metavar="DIR",
                    help="write what the timed path computed in its last step to DIR/<name>.npy (float32; the parameters "
                         "after the step as a fixed seeded sample), so that two builds can be compared output for output")
    ap.add_argument("--scaling", choices=["weak", "strong"], default="weak",
                    help="weak: every rank renders its own --batch rays (global batch = batch x N); strong: the --batch "
                         "rays of a step are split over the ranks (SURVEY.md 8e: same draw on all ranks, contiguous slices)")
    a = ap.parse_args()
    if a.steps < 1 or a.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if a.envmap_h is None:
        a.envmap_h, a.envmap_w = (8, 16) if a.config == 3 else (16, 32)
    return a


class Args:   # the three fields render_with_BRDF reads from the train scripts' namespace (opt.py:150-154)
    second_nSample, second_near, second_far = 96, 0.05, 1.5


L1_WEIGHT = 4e-5      # L1_weight_rest (configs/single_light/armadillo.txt)


def loss_of(ret, target, model, it=0, l1_in_optimizer=False):
    """Loss assembly of the relight phase, train_tensoIR.py:262-312 (TV is switched off once relight starts,
    :396-399; weights from configs/single_light/armadillo.txt).  With ``l1_in_optimizer`` the L1_weight_rest *
    density_L1 term is applied by tensoir_b200.optim.FusedAdam (same gradient, folded into the optimiser pass)."""
    loss = torch.mean((ret['rgb_map'] - target) ** 2)
    if not l1_in_optimizer:
        loss = loss + L1_WEIGHT * model.density_L1()
    loss = loss + 0.2 * torch.mean((ret['rgb_with_brdf_map'] - target) ** 2)
    loss = loss + 0.0005 * ret['normals_diff_map'].mean() + 0.001 * ret['normals_orientation_loss_map'].mean()
    loss = loss + 0.001 * ret['roughness_smoothness_loss'] + 0.001 * ret['albedo_smoothness_loss']
    return loss


class ClockSampler:
    """nvidia-smi sampled DURING the timed region (B200_PROFILING.md clocks line)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index, period_ms=50):
        self.rows, self.stamps, self.proc, self.idx, self.period = [], [], None, gpu_index, period_ms
        self.begin = None

    def start(self):
        """Spawn the sampler (idempotent).  Called BEFORE the warm-up steps so that nvidia-smi's own start-up (100+ ms,
        longer than a 20-step timed region of this bench) is over when the timed region begins."""
        if self.proc is not None:
            return
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.idx), "-lms", str(self.period)], stdout=subprocess.PIPE,
                                         text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def mark(self):
        """The timed region starts now: rows that arrive from here on are the ones reported."""
        self.start()
        if self.begin is None:
            self.begin = time.monotonic()

    def _read(self):
        for line in self.proc.stdout:
            self.stamps.append(time.monotonic())
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        end = time.monotonic()
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        self.t.join(timeout=2)
        begin = self.begin if self.begin is not None else 0.0
        inside = [r for r, ts in zip(self.rows, self.stamps) if begin <= ts <= end + 0.05]
        # rows before mark() were taken during the warm-up steps (same load); used only if none fell inside
        rows, window = (inside, "timed") if inside else (self.rows, "warmup+timed")
        sm = sorted(float(r[1]) for r in rows if len(r) > 2 and r[1].replace('.', '').isdigit())
        mx = [float(r[2]) for r in rows if len(r) > 2 and r[2].replace('.', '').isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            for j, nm in enumerate(names):
                if len(r) > 5 + j and r[5 + j].lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "window": window, "period_ms": self.period}


def dist_setup(n):
    if n > 1 or "RANK" in os.environ:
        rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
        local = int(os.environ.get("LOCAL_RANK", rank))
        return rank, world, local
    return 0, 1, 0


# ---------------------------------------------------------------------------------------------------------------
def run_reference(a, rank, world):
    """The reference's own algorithm on the host CPU cores (oracle port), bounded sample per step."""
    if rank != 0:
        return
    out = cpu_baseline(a, steps=a.steps, warmup=a.warmup, budget_s=240.0)
    line = {"metric": METRIC, "value": out["value"], "unit": UNIT, "n_gpus": a.gpus, "steps": out["steps_done"],
            "warmup": a.warmup, "ms_per_step": out["ms_per_step"], "higher_is_better": True, "scaling": a.scaling,
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "impl": "reference",
            "config": workload_config(a, parallelism=f"cpu{out['cores']}"),
            "cpu_baseline": {"value": out["value"], "unit": UNIT, "cores": out["cores"], "kind": "port",
                             "sample": out["sample"]},
            "e2e": {"value": out["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


def workload_config(a, parallelism):
    from tensoir_b200.synthetic import n_samples_for
    cfg = getattr(a, "config", 2)
    what = WORKLOADS[cfg].format(grid=a.grid, dirs=f"{getattr(a, 'envmap_h', 16)}x{getattr(a, 'envmap_w', 32)} = "
                                                   f"{getattr(a, 'envmap_h', 16) * getattr(a, 'envmap_w', 32)}")
    return {"workload": f"relight training step, lego-shaped synthetic scene ({what}): "
                        f"TensorVMSplit {a.grid}^3 (16/48 comps, 3 MLP heads, SG light), batch {a.batch} rays of "
                        f"100 views 800x800, N_samples {n_samples_for(a.grid)}, {getattr(a, 'envmap_h', 16)}x"
                        f"{getattr(a, 'envmap_w', 32)} stratified secondary dirs x 96 samples, fwd+bwd+Adam (one fused pass incl. the L1 regulariser)",
            "global_batch_rays": a.batch * (max(1, a.gpus) if getattr(a, "scaling", "weak") == "weak" else 1),
            "grid": a.grid, "parallelism": parallelism,
            "l2": "inputs change every step (new ray batch, updated parameters); VM tensors "
                  f"({'exceed' if a.grid >= 256 else 'fit in'} L2 at this grid)"}


def make_lego_state(grid, seed=20211202):
    """CPU-side twin of tensoir_b200.synthetic.make_lego_model for the CPU baseline: the same field (same seed, same
    init order, built with the host classes on the CPU - no kernels run) handed to the oracle as an OracleField, with
    the alpha mask computed by the oracle itself.  Lives here (not in the package) because only bench.py / tests may
    touch oracle/."""
    from oracle import tensoir_oracle as O
    from tensoir_b200.synthetic import install_lego_density
    from tensoir_b200.tensorf import TensorVMSplit
    torch.manual_seed(seed)
    aabb = torch.tensor([[-1.5] * 3, [1.5] * 3])
    m = TensorVMSplit(aabb, [grid] * 3, 'cpu', density_n_comp=[16] * 3, appearance_n_comp=[48] * 3, app_dim=27,
                      near_far=[2.0, 6.0], shadingMode='MLP_Fea', alphaMask_thres=0.001, density_shift=-10,
                      distance_scale=25, pos_pe=2, view_pe=2, fea_pe=2, featureC=128, step_ratio=0.5,
                      fea2denseAct='softplus', normals_kind='derived_plus_predicted', light_rotation=["000"],
                      light_kind='sg', numLgtSGs=128)
    install_lego_density(m)
    f = O.field_from_state_dict(m.state_dict(), aabb, [grid] * 3, kind="rotated", light_rotation=[0])
    r = min(grid, 256)
    O.update_alpha_mask(f, (r, r, r))
    return f


def _pick_threads(f, n_s):
    """torch CPU ops on the oracle's small tensors get SLOWER past some thread count (on the 128-core GPU host a step
    takes minutes at 128 threads); probe a few counts with one small secondary march each and keep the fastest -
    i.e. all the threads the reference can actually use."""
    from oracle import tensoir_oracle as O
    cpu = os.cpu_count() or 1
    cands = sorted({c for c in (cpu, 64, 32, 16, 8) if c <= cpu}, reverse=True)
    g = torch.Generator().manual_seed(1)
    pts = (torch.rand(4096, 3, generator=g) * 2 - 1) * 0.9
    dirs = torch.nn.functional.normalize(torch.randn(4096, 3, generator=g), dim=-1)
    li = torch.zeros(4096, 1, dtype=torch.int32)
    best, probe = None, {}
    for c in cands:
        torch.set_num_threads(c)
        O.compute_radiance(f, pts[:256], dirs[:256], li[:256], 96, 0.05, 1.5)          # warm
        t0 = time.perf_counter()
        O.compute_radiance(f, pts, dirs, li, 96, 0.05, 1.5)
        probe[c] = time.perf_counter() - t0
        if best is None or probe[c] < probe[best]:
            best = c
        if probe[c] > 20.0:          # hopeless setting, do not waste the budget on slower ones
            continue
    torch.set_num_threads(best)
    return best, probe


def cpu_baseline(a, steps=2, warmup=1, budget_s=120.0):
    """Oracle (port of the reference) fwd+bwd+Adam on a bounded sample of the same workload, host cores only."""
    from oracle import tensoir_oracle as O
    from tensoir_b200.synthetic import hemisphere_poses, training_batch, n_samples_for
    torch.set_num_threads(min(os.cpu_count() or 1, 32))
    f = make_lego_state(a.grid)
    n_s = n_samples_for(a.grid)
    cores, probe = _pick_threads(f, n_s)
    for p in f.parameters():
        p.requires_grad_(True)
    opt = torch.optim.Adam([{"params": f.parameters(), "lr": 1e-3}], betas=(0.9, 0.99))
    poses = hemisphere_poses(100)
    rays_total, t_total, done = 0, 0.0, 0
    t_begin = time.perf_counter()
    for it in range(warmup + steps):
        rays, li = training_batch(poses, a.cpu_rays, it)
        f.counters.clear()
        t0 = time.perf_counter()
        ret = O.renderer_train(f, rays, li, n_s, True, True, True, 'stratified_sampling', 160000, 96, 0.05, 1.5)
        target = torch.full_like(ret["rgb_map"], 0.5)
        loss = torch.mean((ret['rgb_map'] - target) ** 2) + 0.2 * torch.mean((ret['rgb_with_brdf_map'] - target) ** 2)
        loss = loss + 0.0005 * ret['normals_diff_map'].mean() + 0.001 * ret['normals_orientation_loss_map'].mean()
        loss = loss + 0.001 * ret['roughness_smoothness_loss'] + 0.001 * ret['albedo_smoothness_loss']
        opt.zero_grad()
        loss.backward()
        opt.step()
        dt = time.perf_counter() - t0
        if it >= warmup:
            rays_total += a.cpu_rays + f.counters.get("secondary_rays", 0)
            t_total += dt
            done += 1
        if time.perf_counter() - t_begin > budget_s and done >= 1:
            break
    return {"value": rays_total / t_total, "ms_per_step": 1e3 * t_total / max(done, 1), "cores": cores,
            "steps_done": done,
            "sample": f"{a.cpu_rays} primary rays/step x {done} steps of the same workload (oracle port, torch CPU, "
                      f"{cores} of {os.cpu_count()} threads = fastest of the probed counts "
                      f"{ {k: round(v, 2) for k, v in probe.items()} } s)"}


# ---------------------------------------------------------------------------------------------------------------
WORKLOADS = {
    2: "BASELINE configs[1] shape: single light, TensorVMSplit {grid}^3, 16x32 stratified secondary dirs",
    3: "BASELINE configs[2] shape: multi_light_rotated (3 rotations of one light), {dirs} stratified secondary dirs per "
       "surface sample",
    4: "BASELINE configs[3] shape: multi_light_general (TensorVMSplit with light_name_list of 3), {grid}^3",
    5: "BASELINE configs[4] shape: relight_importance pass, 2048x1024 synthetic HDR env map(s), 512 importance samples, "
       "visibility through the density march",
}


def build_model(a, dev):
    from tensoir_b200.synthetic import make_lego_model
    with contextlib.redirect_stdout(sys.stderr):     # stdout carries exactly one line: the JSON result
        if a.config == 3:
            return make_lego_model(a.grid, dev, lights=("000", "120", "240"), envmap=(a.envmap_h, a.envmap_w)), 3
        if a.config == 4:
            return make_lego_model(a.grid, dev, lights=("sunset", "snow", "courtyard"), general=True), 3
        return make_lego_model(a.grid, dev), 1


def measure(a, model, n_lights, rank, world, local, dev, scaling, with_e2e, clocks=None):
    """Device-resident (and optionally end-to-end) timed regions of the training step for one scaling mode."""
    from tensoir_b200 import Renderer_TensoIR_train, _lib, ops
    from tensoir_b200.dp import GradBucket, shard_batch
    from tensoir_b200.synthetic import hemisphere_poses, training_batch, n_samples_for
    params = []
    for grp in model.get_optparam_groups(0.02, 0.001):
        gp = grp["params"]
        params += [gp] if isinstance(gp, torch.Tensor) else list(gp)     # a bare Parameter must not be iterated
    # same optimiser and hyper-parameters as train_tensoIR.py:206; fused=True selects PyTorch's single-kernel
    # multi-tensor implementation of the identical update (SURVEY.md §8f item 3)
    fused_opt = not a.torch_adam
    if fused_opt:
        # tensoir_b200.optim.FusedAdam: the same Adam update in one launch over all parameters, + the density L1
        # regulariser's gradient + clearing the gradients (SURVEY.md 8 f3)
        from tensoir_b200.optim import FusedAdam
        from tensoir_b200.static_step import lr_tensors
        groups = model.get_optparam_groups(0.02, 0.001)
        opt = FusedAdam(groups if a.eager else lr_tensors(groups, dev), betas=(0.9, 0.99))
        opt.density_l1(model, L1_WEIGHT)
    else:
        opt = torch.optim.Adam(model.get_optparam_groups(0.02, 0.001), betas=(0.9, 0.99), fused=True,
                               capturable=not a.eager)
    bucket = GradBucket(params) if world > 1 else None
    poses = hemisphere_poses(100)
    n_s = n_samples_for(a.grid)
    total = a.warmup + a.steps
    if scaling == "weak":
        # every rank draws its own 4096-ray batch each step (global batch = batch * world)
        per_rank = a.batch
        host_batches = [training_batch(poses, a.batch, it * world + rank, n_lights=n_lights) for it in range(2 * total)]
    else:
        # the same global batch on every rank (same seed), rank r keeps its contiguous slice (SURVEY.md 8e)
        lo, hi = shard_batch(a.batch, rank, world)
        per_rank = hi - lo
        host_batches = [tuple(t[lo:hi].contiguous() for t in training_batch(poses, a.batch, it, n_lights=n_lights))
                        for it in range(2 * total)]
    pinned = [(r.pin_memory(), l.pin_memory()) for r, l in host_batches]
    target = torch.full((per_rank, 3), 0.5, device=dev)
    counters = ops.new_counters(dev)
    model.__dict__["_tir_counters"] = counters
    last = {}          # the renderer's outputs and the loss of the most recent step

    def loss_fn(ret, m):
        last["ret"] = ret
        return loss_of(ret, target, m, l1_in_optimizer=fused_opt)
    # production mode of the marches: work that would only feed the mask / density COUNTERS is skipped (the rest of a ray
    # whose transmittance is exactly 0); rays, appearance samples and every output are unaffected.
    model.__dict__["_tir_lean"] = True

    graphed = None
    if not a.eager:
        # whole-step CUDA graph: static-capacity sample lists, host randoms staged into device buffers, replay
        from tensoir_b200.static_step import StaticTrainStep
        # a replay rewrites the tensors the captured loss_fn saw: last["ret"] then holds the latest replay's outputs
        graphed = StaticTrainStep(model, opt, per_rank, n_s, Args, loss_fn, grad_bucket=bucket, device=dev)
        # lists sized from 8 batches x 1.5; they grow by themselves (high-water marks, re-capture) and a replay whose
        # lists did not fit is an exact no-op that is redone (static_step.py) - never a silently different step
        graphed.calibrate(host_batches[:8])
        graphed.capture(warmup=3)

    def step(rays, li):
        if graphed is not None:
            last["loss"] = graphed.run(rays, li)
            return last["loss"]
        ret = Renderer_TensoIR_train(rays, None, li, model, N_samples=n_s, white_bg=True, is_train=True,
                                     is_relight=True, sample_method='stratified_sampling', chunk_size=160000,
                                     device=dev, args=Args)
        loss = loss_fn(ret, model)
        opt.zero_grad(set_to_none=False)
        loss.backward()
        if bucket is not None:
            bucket.all_reduce_mean()
        opt.step()
        last["loss"] = loss
        return loss

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed_region(batches, read_loss):
        counters.zero_()
        launches0 = _lib.launch_count
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.profiler.start()               # no-op unless a profiler is attached with --profile-from-start off
        e0.record()
        for rays, li in batches:
            loss = step(rays, li)
            if read_loss:
                loss.item()                       # device -> host read of the step's result
        e1.record()
        barrier()
        torch.cuda.profiler.stop()
        ms = e0.elapsed_time(e1)
        if graphed is not None:
            graphed.flush()                       # settle the last replays: overflowed ones would be redone here
        t = torch.tensor([ms], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        c = counters.clone()
        if world > 1:
            dist.all_reduce(c, op=dist.ReduceOp.SUM)
        return float(t.item()), ops.counters_dict(c), _lib.launch_count - launches0

    # ---- device-resident arm: inputs already in HBM when the timed region starts
    dev_batches = [(r.to(dev), l.to(dev)) for r, l in host_batches[:total]]
    if clocks is not None:
        clocks.start()
    for rays, li in dev_batches[:a.warmup]:
        step(rays, li)
    if graphed is not None:
        # lists at 4x the longest seen during warm-up (every list kernel works on the device-side length, so padding is
        # nearly free): the gray-target training of this bench grows the appearance list by tens of percent per 10 steps
        graphed.reserve(4.0)
        sys.stderr.write(f"bench[{scaling}]: static lists {graphed.capacities()} after warm-up (seen {graphed._seen})\n")
    if clocks is not None:
        clocks.mark()
    events0 = (graphed.redone, graphed.recaptures) if graphed is not None else (0, 0)
    ms, cnt, launches = timed_region(dev_batches[a.warmup:], read_loss=False)
    out = {"scaling": scaling, "ms": ms, "cnt": cnt, "launches": launches, "per_rank": per_rank,
           "value": cnt["rays"] / (ms * 1e-3),   # TIR_CNT_RAYS counts every marched ray: primary + secondary
           "last_batch": dev_batches[-1], "n_s": n_s}
    if a.dump_outputs is not None and rank == 0:
        # before the end-to-end arm trains the model further
        out["outputs"] = train_step_outputs(last["ret"], last["loss"], model)
    if with_e2e:
        # ---- end-to-end arm: pinned HOST buffers through the public boundary, loss read back every step.
        # Default: the host sends (view, pixel, light) ids - 12 B/ray - and the rays are generated on the device
        # (ops.generate_rays, SURVEY.md 8 f4); --host-rays sends the 28 B/ray the reference's loop indexes from its table.
        if a.host_rays:
            e2e_batches = pinned
            out["e2e_inputs"] = "rays [n,6] fp32 + light_idx from pinned host memory"
            out["h2d_per_ray"] = 28
        else:
            from tensoir_b200.synthetic import training_batch_ids
            poses_dev = poses.to(dev)
            slice_ = slice(None) if scaling == "weak" else slice(*shard_batch(a.batch, rank, world))
            ids = [training_batch_ids(poses.shape[0], a.batch, (it * world + rank) if scaling == "weak" else it,
                                      n_lights=n_lights) for it in range(2 * total)]
            ids = [tuple(t[slice_].contiguous().pin_memory() for t in trip) for trip in ids]

            class _Ids:                      # looks like a (rays, light_idx) pair to step(): rays built on the device
                def __init__(self, trip):
                    self.trip = trip

                def __iter__(self):
                    v, p, l = (t.to(dev, non_blocking=True) for t in self.trip)
                    return iter((ops.generate_rays(poses_dev, v, p), l))
            e2e_batches = [_Ids(t) for t in ids]
            out["e2e_inputs"] = "(view, pixel, light) ids from pinned host memory, rays generated on the device"
            out["h2d_per_ray"] = 12
        for rays, li in e2e_batches[total:total + a.warmup]:
            step(rays, li)
        ms_e2e, cnt_e2e, _ = timed_region(e2e_batches[total + a.warmup:2 * total], read_loss=True)
        out.update(ms_e2e=ms_e2e, e2e_value=cnt_e2e["rays"] / (ms_e2e * 1e-3))
    out["clocks"] = clocks.stop() if clocks is not None else None
    events1 = (graphed.redone, graphed.recaptures) if graphed is not None else (0, 0)
    overflow = graphed.overflowed() if graphed is not None else 0
    out.update(caps=graphed.capacities() if graphed is not None else None, overflow=overflow, events=events1)
    if graphed is not None:
        graphed.release()
    model.__dict__.pop("_tir_counters", None)
    bad = torch.tensor([float(events1 != events0 or overflow > 0)], device=dev)
    if world > 1:
        dist.all_reduce(bad, op=dist.ReduceOp.MAX)
    if bad.item() > 0:
        # a timed replay overflowed its static lists (it was a no-op and was redone) or the graph had to be re-captured
        # inside the timed region: the K timed steps are not K clean steps -> no number
        sys.stderr.write(f"bench: static lists overflowed / re-captured inside the timed region on rank {rank} "
                         f"(redone, recaptures) {events0} -> {events1}, overflowed replays {overflow}; no result\n")
        sys.stderr.flush()
        if world > 1:
            torch.cuda.synchronize()
            dist.barrier()
        os._exit(3)
    return out


def torch_gpu_reference(a, model, n_lights):
    """The unmodified reference (the checkout given by --reference) on the same GPU / field / batches, in a subprocess
    (its `models` and `renderer` modules must not meet tensoir_b200's).  None without --reference."""
    ref = a.reference and os.path.abspath(a.reference)
    if not ref or a.config not in (2, 3) or (a.envmap_h, a.envmap_w) != (16, 32):
        return None          # (the reference's checkpoint kwargs carry no envmap size: only its 16x32 default is comparable)
    import tempfile
    tmp = tempfile.mkdtemp(prefix="tir_ref_")
    ckpt = os.path.join(tmp, "field.th")
    model.save(ckpt)
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([os.path.join(ROOT, "tools", "ref_stubs"), ref, ROOT]))
    for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK", "MASTER_ADDR", "MASTER_PORT"):
        env.pop(k, None)
    try:
        p = subprocess.run([sys.executable, "-P", os.path.join(ROOT, "tools", "ref_torch_gpu.py"), "--ckpt", ckpt,
                            "--grid", str(a.grid), "--batch", str(a.batch), "--n_lights", str(n_lights)], cwd=ref, env=env,
                           capture_output=True, text=True, timeout=600)
        lines = [l for l in p.stdout.splitlines() if l.startswith("{")]
        if p.returncode != 0 or not lines:
            return {"unavailable": (p.stderr or p.stdout)[-300:]}
        return json.loads(lines[-1])
    except Exception as e:      # the denominator is optional context, never a reason to lose the bench line
        return {"unavailable": repr(e)[:300]}
    finally:
        import shutil
        shutil.rmtree(tmp, ignore_errors=True)


def main():
    a = parse()
    rank, world, local = dist_setup(a.gpus)
    if a.impl == "reference":
        run_reference(a, rank, world)
        return
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback for the product path)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    import __graft_entry__ as g
    if rank == 0:
        g.build()
    if world > 1:
        dist.barrier()
    from tensoir_b200 import _lib
    from tensoir_b200.dp import broadcast_parameters
    _lib.load()
    if a.config == 5:
        run_relight_pass(a, rank, world, local, dev)
        return

    model, n_lights = build_model(a, dev)
    broadcast_parameters(model.parameters())
    ref_gpu = torch_gpu_reference(a, model, n_lights) if (rank == 0 and world == 1 and not a.no_torch_reference) else None
    clocks = ClockSampler(local) if rank == 0 else None
    m = measure(a, model, n_lights, rank, world, local, dev, a.scaling, with_e2e=True, clocks=clocks)
    strong = None
    if world > 1 and a.scaling == "weak" and not a.no_strong:
        # the north-star's strong-scaling number in the same run: ONE --batch-ray batch split over the ranks
        strong = measure(a, model, n_lights, rank, world, local, dev, "strong", with_e2e=False)

    def finish():
        """Leave together: a CUDA graph holding NCCL kernels plus communicator teardown can hang at interpreter exit,
        so every rank meets at one last barrier and exits without running destructors."""
        sys.stdout.flush()
        sys.stderr.flush()
        if world > 1:
            torch.cuda.synchronize()
            dist.barrier()
            os._exit(0)

    if rank != 0:
        finish()
        return

    ms, cnt, per_rank = m["ms"], m["cnt"], m["per_rank"]
    # ---- roofline of the dominant kernel (the secondary march), timed live with CUDA events on the launch stream
    roof = roofline(model, m["last_batch"], m["n_s"], dev, a)
    line = {"metric": METRIC, "value": m["value"], "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": ms / a.steps, "higher_is_better": True, "scaling": a.scaling, "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": workload_config(a, f"dp{world}"),
            "primary_rays_per_s": per_rank * a.steps * world / (ms * 1e-3),
            "secondary_rays_per_s": (cnt["rays"] - per_rank * a.steps * world) / (ms * 1e-3),
            "counters_per_step": {k: v / a.steps for k, v in cnt.items()},
            "e2e": {"value": m["e2e_value"], "unit": UNIT, "ms_per_step": m["ms_e2e"] / a.steps,
                    "inputs": m["e2e_inputs"],
                    # ray inputs + the host-drawn per-ray jitter and stratified light directions
                    "h2d_bytes_per_step": (per_rank * m["h2d_per_ray"] + per_rank * 4 + a.envmap_h * a.envmap_w * 3 * 4) * world,
                    "d2h_bytes_per_step": 4 * world},
            "counters_note": "mask / density are the queries actually made (TIR_MARCH_LEAN_COUNTERS: the rest of a ray "
                             "whose transmittance is exactly 0 is skipped); rays / app are the reference's counts",
            "gpu_launches": m["launches"], "clocks": m["clocks"], "roofline": roof,
            "execution": ("eager" if a.eager else f"cuda-graph replay of the whole step (static list capacities "
                          f"{m['caps']}, overflowed steps: {m['overflow']}, redone: {m['events'][0]}, re-captures during "
                          f"warm-up: {m['events'][1]}; an overflowed replay is a device-side no-op that is redone with "
                          f"larger lists)")}
    if strong is not None:
        line["strong_scaling"] = {"what": f"same run, ONE {a.batch}-ray batch per step split over the {world} ranks "
                                          f"(contiguous slices, same draw everywhere), one gradient all-reduce per step",
                                  "value": strong["value"], "unit": UNIT, "ms_per_step": strong["ms"] / a.steps,
                                  "global_batch_rays": a.batch, "rays_per_rank": strong["per_rank"]}
    if ref_gpu is not None:
        if "ms_per_step" in ref_gpu:
            ref_gpu["speedup_ms_per_step"] = ref_gpu["ms_per_step"] / (ms / a.steps)
        line["torch_gpu_reference"] = ref_gpu
    if a.dump_outputs is not None:
        write_outputs(a.dump_outputs, m["outputs"])
    if not a.no_cpu_baseline and world == 1:
        cb = cpu_baseline(a, steps=2, warmup=1)
        line["cpu_baseline"] = {"value": cb["value"], "unit": UNIT, "cores": cb["cores"], "kind": "port",
                                "sample": cb["sample"]}
    print(json.dumps(line))
    finish()


def train_step_outputs(ret, loss, model, n_sample=1 << 16, seed=0):
    """What a caller of the training step receives from its last call, as float32 arrays: the loss, every tensor the
    renderer returned, and each parameter after the optimiser step - all of a small one, a fixed seeded sample of
    ``n_sample`` entries (the same positions in every run) of a larger one."""
    out = {"loss": loss}
    out.update((k, v) for k, v in ret.items() if torch.is_tensor(v))
    g = torch.Generator().manual_seed(seed)
    for k, p in model.named_parameters():
        flat = p.detach().reshape(-1)
        if flat.numel() > n_sample:
            flat = flat[torch.randperm(flat.numel(), generator=g)[:n_sample].sort().values.to(flat.device)]
        out["param." + k] = flat
    return {k: v.detach().float().cpu().numpy() for k, v in out.items()}


def write_outputs(path, arrays, limit=64 << 20):
    """DIR/<name>.npy for every array; refuses to write more than ``limit`` bytes in all."""
    import numpy as np
    total = sum(v.nbytes for v in arrays.values())
    if total > limit:
        raise SystemExit(f"--dump-outputs: {total} bytes of outputs exceed the {limit}-byte limit")
    os.makedirs(path, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(path, k + ".npy"), np.ascontiguousarray(v))


def synthetic_hdr(h=1024, w=2048, seed=20211202):
    """Log-normal radiance plus one bright sun disc (SURVEY.md 8d, config 5)."""
    g = torch.Generator().manual_seed(seed)
    env = torch.exp(0.6 * torch.randn(h // 16, w // 16, 3, generator=g)).permute(2, 0, 1)[None]
    env = torch.nn.functional.interpolate(env, size=(h, w), mode="bilinear", align_corners=False)[0].permute(1, 2, 0)
    yy, xx = torch.meshgrid(torch.arange(h), torch.arange(w), indexing="ij")
    sun = ((yy - h // 4) ** 2 + (xx - w // 3) ** 2) < (h // 40) ** 2
    env = env * 0.5
    env[sun] = 400.0
    return env.contiguous().numpy()


def run_relight_pass(a, rank, world, local, dev):
    """BASELINE configs[4]: scripts/relight_importance.py's pass. A step = one 4096-ray chunk of a test view: primary
    march (eval) + 512 importance-sampled light directions per surface hit, visibility through the density march, GGX,
    pdf-weighted mean, sRGB, background lookup.  Test views are sharded over the ranks (no data-path collective)."""
    from tensoir_b200 import ops
    from tensoir_b200.relight import Environment_Light, relight_chunk
    from tensoir_b200.synthetic import hemisphere_poses, image_rays
    model, _ = build_model(a, dev)
    env = Environment_Light({"synthetic": synthetic_hdr()}, device=dev)
    poses = hemisphere_poses(200)
    total = a.warmup + a.steps
    # object-centred 400 x 320 window of the view: 31 chunks of 4096 rays with similar content, so that the warm-up sees
    # the tensor sizes of the timed steps (a chunk with more hits than any warm-up chunk would time the caching
    # allocator's cudaMalloc, not the pass)
    view = image_rays(poses[7 + rank]).reshape(800, 800, 6)[240:560, 200:600].reshape(-1, 6)
    n_chunks = view.shape[0] // a.batch
    if total > n_chunks:
        raise SystemExit(f"--config 5: warmup + steps must be <= {n_chunks}")
    # heaviest chunks first in the warm-up: order by distance from the image centre row
    order = sorted(range(n_chunks), key=lambda i: abs(i - n_chunks // 2))
    chunks = [view[i * a.batch:(i + 1) * a.batch].contiguous() for i in order[:total]]
    pinned = [c.pin_memory() for c in chunks]
    counters = ops.new_counters(dev)
    model.__dict__["_tir_counters"] = counters
    host_out = torch.empty(a.batch, 3).pin_memory()

    @torch.no_grad()
    def step(rays_in, read_back):
        rays = rays_in.to(dev, non_blocking=True)
        li = torch.zeros(rays.shape[0], 1, dtype=torch.int32, device=dev)
        rgb, depth, normal, albedo, rough, fresnel, acc, *_ = model(rays, li, is_train=False, white_bg=True,
                                                                    ndc_ray=False, N_samples=-1)
        img, _ = relight_chunk(model, env, "synthetic", rays, (depth, normal, albedo, rough.repeat(1, 3), fresnel, acc),
                               1.0, None, 512)
        if read_back:
            host_out.copy_(img, non_blocking=True)
            torch.cuda.current_stream().synchronize()
        return img

    def timed(batches, read_back):
        counters.zero_()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for c in batches:
            last["img"] = step(c, read_back)
        e1.record()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t = torch.tensor([e0.elapsed_time(e1)], device=dev)
        c = counters.clone()
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dist.all_reduce(c, op=dist.ReduceOp.SUM)
        return float(t.item()), ops.counters_dict(c)

    last = {}
    dev_chunks = [c.to(dev) for c in chunks[:total]]
    clocks = ClockSampler(local) if rank == 0 else None
    if clocks is not None:
        clocks.start()
    for c in dev_chunks[:a.warmup]:
        step(c, False)
    if clocks is not None:
        clocks.mark()
    ms, cnt = timed(dev_chunks[a.warmup:], False)
    if a.dump_outputs is not None and rank == 0:
        write_outputs(a.dump_outputs, {"relit_rgb": last["img"].float().cpu().numpy()})
    for c in pinned[:a.warmup]:
        step(c, True)
    ms_e2e, cnt_e2e = timed(pinned[a.warmup:total], True)
    clk = clocks.stop() if clocks is not None else None
    if rank != 0:
        if world > 1:
            torch.cuda.synchronize(); dist.barrier(); os._exit(0)
        return
    # roofline of the dominant kernel: the visibility march (density only) over the chunk's (hit, light sample) rays
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    peak = json.load(open(peaks_path))["hbm_gbs"] if os.path.exists(peaks_path) else 6650.0
    bytes_alg = 32 * cnt["mask"] + 1152 * cnt["density"] + 16 * (cnt["rays"] - a.batch * a.steps * world)
    line = {"metric": METRIC.replace("relight training step", "relight_importance pass"), "value": cnt["rays"] / (ms * 1e-3),
            "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup, "ms_per_step": ms / a.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOADS[5] + f"; TensorVMSplit {a.grid}^3, {a.batch}-ray chunks of 800x800 test views "
                                                  f"sharded over {world} rank(s), 1 env map", "grid": a.grid,
                       "parallelism": f"views{world}"},
            "counters_per_step": {k: v / a.steps for k, v in cnt.items()},
            "e2e": {"value": cnt_e2e["rays"] / (ms_e2e * 1e-3), "unit": UNIT, "ms_per_step": ms_e2e / a.steps,
                    "h2d_bytes_per_step": a.batch * 24 * world, "d2h_bytes_per_step": a.batch * 12 * world},
            "gpu_launches": int(_launches_since_start()), "clocks": clk,
            "roofline": {"bound": "hbm", "kernel": "march_kernel<16,TABLE,density-only> (visibility rays)",
                         "note": "step-level: algorithmic bytes of all marches of the step / step time (the visibility "
                                 "march is ~all of it)", "achieved": bytes_alg / a.steps / (ms / a.steps * 1e-3) / 1e9,
                         "peak": peak, "unit": "GB/s", "frac": bytes_alg / (ms * 1e-3) / 1e9 / peak, "traffic": None}}
    print(json.dumps(line))
    if world > 1:
        torch.cuda.synchronize(); dist.barrier(); os._exit(0)


def _launches_since_start():
    from tensoir_b200 import _lib
    return _lib.launch_count


def roofline(model, batch, n_s, dev, a):
    """achieved = algorithmic bytes / launch duration of the secondary march kernel (SURVEY.md §8d:
    32 B per alpha-mask query + 1152 B per density sample + 16 B out per ray), CUDA events, after warm-up."""
    from tensoir_b200 import ops
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, src = json.load(open(peaks_path))["hbm_gbs"], "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
    else:
        peak, src = 6650.0, "fallback (B200_PROFILING.md)"
    rays, li = batch
    with torch.no_grad():
        out = model(rays, li, is_train=False, is_relight=True, N_samples=n_s)
    depth, normal, acc_mask = out[1], out[2], out[9]
    surf = (rays[:, :3] + depth[:, None] * rays[:, 3:])[acc_mask]
    dirs = model.gen_light_incident_dirs(method='stratified_sampling').to(dev)
    st = ops.SecondaryStages(model, surf, normal[acc_mask], li[acc_mask], dirs)          # timed: production (lean) mode
    lean = model.__dict__.pop("_tir_lean", False)
    st_count = ops.SecondaryStages(model, surf, normal[acc_mask], li[acc_mask], dirs)    # counts: the reference's work
    model.__dict__["_tir_lean"] = lean

    def t(fn, n=10):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / n
    ms_march = t(st.march)
    st.march()
    c_run = ops.counters_dict(st.counters)        # units the timed (production / lean) launch actually processed
    ms_full = t(st_count.march)                   # the same kernel evaluating everything the reference evaluates
    st_count.march()
    c = ops.counters_dict(st_count.counters)      # the reference algorithm's counts (count-parity mode)
    ms_mlp = t(st.mlp)
    b_run = 32 * c_run["mask"] + 1152 * c_run["density"] + 16 * c_run["rays"]
    b_full = 32 * c["mask"] + 1152 * c["density"] + 16 * c["rays"]
    traffic, traffic_src = None, None
    summary = os.path.join(ROOT, "profiles", "r2_ncu_march_raw_summary.csv")
    if os.path.exists(summary):          # dram bytes of the same kernel / workload / build, one `ncu --set full` capture
        vals = {}
        for ln in open(summary):
            k, unit, v = (ln.strip().split(",") + ["", ""])[:3]
            if k.startswith("dram__bytes"):
                vals[k] = float(v) * {"Mbyte": 1e6, "Kbyte": 1e3, "Gbyte": 1e9, "byte": 1.0}.get(unit, 1.0)
        if len(vals) == 2:
            traffic = sum(vals.values())
            traffic_src = "profiles/r2_ncu_march_raw_summary.csv (ncu --set full of tools/profile_target.py, this build)"
    b_mlp = 3456 * c["app"]
    flops_mlp = 79712 * c["app"]
    return {"bound": "hbm", "kernel": "march_kernel<16,TABLE,app,dense> (secondary density march + compaction)",
            # the launch that is timed inside the step skips the tail of rays whose transmittance is exactly 0: only the
            # units it really processed are credited (conservative); the count-parity launch is reported next to it
            "achieved": b_run / (ms_march * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
            "frac": b_run / (ms_march * 1e-3) / 1e9 / peak, "peak_source": src, "traffic": traffic,
            "traffic_source": traffic_src,
            "note": "the VM factors and the alpha mask are L2-resident (126 MB L2), so measured DRAM traffic is ~400x "
                    "below the algorithmic bytes; frac is algorithmic bytes / time / measured HBM copy bandwidth",
            "ms_per_launch": ms_march, "algorithmic_bytes_per_launch": b_run,
            "units_per_launch": {"mask_queries": c_run["mask"], "density_samples": c_run["density"], "rays": c_run["rays"]},
            "count_parity_launch": {"ms_per_launch": ms_full, "algorithmic_bytes_per_launch": b_full,
                                    "achieved": b_full / (ms_full * 1e-3) / 1e9,
                                    "frac": b_full / (ms_full * 1e-3) / 1e9 / peak,
                                    "units_per_launch": {"mask_queries": c["mask"], "density_samples": c["density"],
                                                         "rays": c["rays"]}},
            "second_kernel": {"kernel": "app_mlp_tc5_kernel (appearance gather -> basis_mat -> 150-128-128-3 MLP on "
                                        "tcgen05.mma, accumulator + split-BF16 activations in TMEM, fp32 accumulate)",
                              "bound": "L2 gather bandwidth / latency (3456 B per sample from the L2-resident factors)",
                              "ms_per_launch": ms_mlp, "app_samples": c["app"],
                              "achieved_GBps": b_mlp / (ms_mlp * 1e-3) / 1e9,
                              "achieved_TFLOPs": flops_mlp / (ms_mlp * 1e-3) / 1e12}}


if __name__ == "__main__":
    main()
