"""What the unmodified reference computed in the checks that pin the oracle and the host code to it, recorded once by
tests/golden/make_golden_reference_pins.py (tests/golden/reference_pins.npz), and the inputs those checks share with
the recorder: the cases, the dataset facts, the element sample of the arrays recorded in part."""
from __future__ import annotations

import functools
import json
import os

import numpy as np
import torch

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_pins.npz")

DS = {"num_keyframes": 12, "num_frames": 50, "near": 0.5, "far": 10.0, "depth_range": [0.5, 10.0], "name": "x", "collection": "y"}
# dataset facts only some constructors read (voxel.py: bbox_min / bbox_max; point.py: total_images_per_frame, val_all)
DS_R2 = dict(DS, bbox_min=[-1.5, -1.25, -1.0], bbox_max=[1.5, 1.25, 1.0], total_images_per_frame=5, val_all=True)
DS_ALPHA = dict(DS, num_keyframes=4, num_frames=6)
FACTS = [
    DS_R2,
    {"num_keyframes": 7, "num_frames": 30, "near": 0.25, "far": 6.0, "depth_range": [0.75, 4.0], "name": "x", "collection": "y",
     "bbox_min": [-0.5, -2.0, -1.5], "bbox_max": [2.5, 1.0, 0.5], "total_images_per_frame": 3, "val_all": False},
]

FRESH_CASES = ["technicolor_trained", "neural3d_trained", "donerf_s16"]
FRESH_RAYS = 777
EDGE_CASES = ["technicolor_trained", "neural3d_trained", "donerf_trained", "immersive_sphere_new", "donerf_cylinder", "technicolor_bbox"]
SHIPPED_GRID = 24 ** 3
REFERENCE_FAILS = ["catacaustics_sphere", "refnerf_sphere", "shiny_z_tensorf", "donerf_z", "shiny_z_depth", "blender_voxel"]
UPSAMPLE_YAMLS = ["technicolor_z_plane", "donerf_sphere"]
REGULARISER_CFG = {"type": "tensorf", "update_AlphaMask_list": [2], "lr_decay_target_ratio": 0.1, "n_iters": 50,
                   "L1_weight_initial": 8e-5, "L1_weight_rest": 4e-5, "TV_weight_density": 0.05, "TV_weight_app": 0.05}
REGULARISER_CALLS = 6
STAGE_YAMLS = ["catacaustics_voxel", "donerf_voxel", "shiny_z_deformable", "immersive_z_plane", "neural_3d_z_plane_static",
               "technicolor_z_plane_no_sample", "shiny_z_plane_cascaded", "shiny_z_plane_feedback", "shiny_z_tensorf_cascaded",
               "technicolor_cascaded"]
ALPHA_CASES = [("technicolor_z_plane", 40000.0), ("donerf_sphere", 40000.0)]
SAMPLED_VALUES = 256  # per-sample points / distances and tables are stored as a fixed sample of this many elements


def flat_sample(numel: int) -> torch.Tensor:
    """The fixed, seeded sample of flat element indices recorded of a large array."""
    g = torch.Generator().manual_seed(1234)
    return torch.randperm(numel, generator=g)[:min(numel, SAMPLED_VALUES)].sort().values


def sampled(key: str, t: torch.Tensor):
    """(recorded values, the same elements of `t`) for an array recorded as a sample; `t` must have the recorded shape."""
    shape = tuple(array(key + "#shape").tolist())
    assert tuple(t.shape) == shape, (key, tuple(t.shape), shape)
    return array(key), t.detach().reshape(-1)[flat_sample(t.numel())]


def corner_occupancy(sd: dict, gain: float) -> dict:
    """Occupancy confined to a corner region, so that the box of occupied voxels is a strict subset of the grid (empty for x
    in the lower half of the box: groups 0 and 1 have x as their planes' column axis, group 2 as its line's axis)."""
    sd = dict(sd)
    for k in list(sd):
        if "density_plane" in k and "time" not in k and sd[k].numel() > 0:
            t = sd[k].clone() * gain
            if not k.endswith(".2"):
                t[..., : t.shape[-1] // 2] = 0
            sd[k] = t
        if "density_line.2" in k and sd[k].numel() > 0:
            t = sd[k].clone()
            t[..., : t.shape[-2] // 2, :] = 0
            sd[k] = t
    return sd


def walk_activations(o, path=""):
    """(path, config) of every `*activation` entry of a config tree."""
    if isinstance(o, dict):
        for k, v in o.items():
            if k.endswith("activation") and (isinstance(v, (dict, str))):
                yield path + "/" + k, v
            if isinstance(v, (dict, list)):
                yield from walk_activations(v, path + "/" + k)
    elif isinstance(o, list):
        for i, v in enumerate(o):
            yield from walk_activations(v, f"{path}[{i}]")


def activation_key(acfg) -> str:
    return json.dumps(acfg, sort_keys=True)


def activation_inputs() -> torch.Tensor:
    return torch.linspace(-6.0, 6.0, 97)


@functools.lru_cache(maxsize=1)
def _load():
    g = np.load(GOLDEN)
    return {k: g[k] for k in g.files if k != "meta_json"}, json.loads(g["meta_json"].tobytes().decode())


def array(key: str) -> torch.Tensor:
    return torch.from_numpy(_load()[0][key].copy())


def keys(prefix: str) -> list:
    return sorted(k for k in _load()[0] if k.startswith(prefix))


def meta(key: str):
    return _load()[1][key]


def model_yamls() -> dict:
    """name -> plain config (None for an empty file) of every model YAML the reference ships, read like Hydra reads it."""
    return meta("model_yamls")
