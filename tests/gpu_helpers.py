"""Build tensoir_b200 models from golden fixtures (GPU tests, smoke, bench)."""
import os
import types

import torch

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load_fixture(name):
    fx = torch.load(os.path.join(GOLDEN, name), weights_only=False)
    if isinstance(fx.get("state_dict"), str):        # a state_dict too large to share the fixture's file
        fx["state_dict"] = torch.load(os.path.join(GOLDEN, fx["state_dict"]), weights_only=True)
    return fx


def renderer_args(n=96, near=0.05, far=1.5):
    a = types.SimpleNamespace()
    a.second_nSample, a.second_near, a.second_far = n, near, far
    return a


def model_from_fixture(fx, device, with_mask=True):
    from tensoir_b200 import TensorVMSplit, TensorVMSplitInit, AlphaGridMask
    aabb = fx["aabb"].to(device)
    common = dict(density_n_comp=[16, 16, 16], appearance_n_comp=[48, 48, 48], app_dim=27, near_far=[2.0, 6.0],
                  shadingMode='MLP_Fea', alphaMask_thres=0.001, density_shift=-10, distance_scale=25, pos_pe=2,
                  view_pe=2, fea_pe=2, featureC=128, step_ratio=0.5, fea2denseAct='softplus')
    if fx["kind"] == "init":
        m = TensorVMSplitInit(aabb, fx["grid_size"], device, **common)
    elif fx["kind"] == "rotated":
        m = TensorVMSplit(aabb, fx["grid_size"], device, normals_kind='derived_plus_predicted',
                          light_rotation=[f"{r:03d}" for r in fx["light_rotation"]], light_kind='sg',
                          numLgtSGs=128, **common)
    else:
        m = TensorVMSplit(aabb, fx["grid_size"], device, normals_kind='derived_plus_predicted',
                          light_name_list=['sunset', 'snow', 'courtyard'], light_kind='sg', numLgtSGs=128, **common)
        for p, v in zip(m.lgtSGs_list, fx["lgt_sgs_list"]):
            p.data.copy_(v.to(device))
    m.load_state_dict({k: v.to(device) for k, v in fx["state_dict"].items()})
    if with_mask:
        m.alphaMask = AlphaGridMask(device, fx["alpha_aabb"].to(device), fx["alpha_volume"].to(device))
    return m
