"""Golden record of what the unmodified reference computes in the checks of tests/test_oracle_vs_reference.py (and the
shipped model YAMLs tests/test_host_logic.py lowers), so that those checks run without a reference checkout.

Recorded, on CPU through oracle/ref_shim.py:
  * every model YAML the reference ships (conf/experiment/model/*.yaml), read like Hydra / OmegaConf reads it, as JSON;
  * rgb (and a fixed sample of rays' points / distances) the reference renders for the seeded cases and YAMLs of the tests;
  * the exception each of the YAMLs the reference cannot run raises inside it;
  * regulariser terms, re-sampled and pruned tables, dense occupancy and alpha masks of the training-schedule checks;
  * the constants the reference's constructors build, and the values of every activation module, for every shipped YAML.

    python tests/golden/make_golden_reference_pins.py
"""
from __future__ import annotations

import copy
import glob
import json
import os
import sys
import types
from types import SimpleNamespace

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

import hyperreel_b200 as hb  # noqa: E402
from hyperreel_b200.config import epochs_to_iters, to_plain  # noqa: E402
from hyperreel_b200.signature import RENDER_ITER, UnsupportedPipeline  # noqa: E402
from hyperreel_b200.state import seeded_state_dict  # noqa: E402
from oracle import ref_shim  # noqa: E402
from tests import reference_pins as P  # noqa: E402
from tests.cases import build_case  # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "reference_pins.npz")


def model_yamls():
    """name -> plain config (None for an empty file), every shipped model YAML."""
    out = {}
    for f in sorted(glob.glob(os.path.join(ref_shim.REFERENCE_ROOT, "conf/experiment/model/*.yaml"))):
        cfg = hb.load_model_yaml(f)
        out[os.path.basename(f)[:-5]] = None if cfg is None else to_plain(cfg)
    return out


def regularizers_package():
    # nlf/regularizers/__init__.py imports every regulariser (and through them the datasets): import tensorf.py alone, with
    # a stand-in for the base class it derives from
    if "nlf.regularizers" not in sys.modules:
        pkg = types.ModuleType("nlf.regularizers")
        pkg.__path__ = [f"{ref_shim.REFERENCE_ROOT}/nlf/regularizers"]
        sys.modules["nlf.regularizers"] = pkg
        base = types.ModuleType("nlf.regularizers.base")
        base.BaseRegularizer = type("BaseRegularizer", (torch.nn.Module,), {})
        sys.modules["nlf.regularizers.base"] = base


def render_ref(plain, ds, sd, rays):
    from nlf.rendering import render_chunked

    ref = ref_shim.build_reference(plain, ds)
    _, unexpected = ref.load_state_dict(sd, strict=False)
    assert not unexpected, unexpected
    with torch.no_grad():
        return render_chunked(rays.clone(), ref, {}, rays.shape[0])["rgb"].reshape(-1, 3)


def main():
    ref_shim.install()
    from nlf.activations import get_activation
    from nlf.rendering import render_chunked

    from tests.test_edge_rays_gpu import craft

    arrays, meta = {}, {}
    yamls = model_yamls()
    meta["model_yamls"] = yamls

    def f32(a):
        return np.ascontiguousarray(torch.as_tensor(a).detach().float().numpy())

    def exact(a):  # compared bit for bit: kept in the reference's own dtype
        return np.ascontiguousarray(torch.as_tensor(a).detach().numpy())

    def put_sampled(key, t):
        t = t.detach()
        arrays[key] = exact(t.reshape(-1)[P.flat_sample(t.numel())])
        arrays[key + "#shape"] = np.array(t.shape, dtype=np.int64)

    # rgb, sample points and distances on fresh rays of the seeded cases
    for name in P.FRESH_CASES:
        case = build_case(name, n=P.FRESH_RAYS)
        ref = ref_shim.build_reference(case.model_cfg_plain, case.dataset)
        ref.load_state_dict(case.state_dict, strict=False)
        out = ref_shim.run_reference(ref, case.rays.clone(), chunk=200, capture=True)
        n = case.rays.shape[0]
        arrays[f"fresh/{name}/rgb"] = f32(out["rgb"])
        put_sampled(f"fresh/{name}/points", out["_embed"]["points"].reshape(n, -1))
        put_sampled(f"fresh/{name}/distances", out["_embed"]["distances"].reshape(n, -1))

    # rgb on the crafted edge rays of tests/test_edge_rays_gpu.py
    for name in P.EDGE_CASES:
        case = build_case(name)
        rays = craft(case)
        ref = ref_shim.build_reference(case.model_cfg_plain, case.dataset)
        ref.load_state_dict(case.state_dict, strict=False)
        with torch.no_grad():
            arrays[f"edge/{name}/rgb"] = f32(render_chunked(rays.clone(), ref, {}, rays.shape[0])["rgb"].reshape(-1, 3))

    # rgb of every shipped YAML that lowers, grid shrunk
    for name, plain in yamls.items():
        if plain is None:
            continue
        cfg = hb.to_cfg(copy.deepcopy(plain))
        cfg.color.net.N_voxel_init = cfg.color.net.N_voxel_final = P.SHIPPED_GRID
        try:
            sig = hb.lower(cfg, P.DS_R2)
        except UnsupportedPipeline:
            continue
        sd = seeded_state_dict(sig, seed=3, density_gain=30.0)
        rays = hb.rays.for_signature(sig, 48, seed=9)
        arrays[f"shipped/{name}/rgb"] = f32(render_ref(to_plain(cfg), P.DS_R2, sd, rays))

    # the YAMLs the reference itself cannot run: the exception it raises
    failures = {}
    for name in P.REFERENCE_FAILS:
        cfg = hb.to_cfg(copy.deepcopy(yamls[name]))
        cfg.color.net.N_voxel_init = cfg.color.net.N_voxel_final = 16 ** 3
        rays = torch.randn(8, 6) * 0.3
        rays[:, 3:6] = torch.nn.functional.normalize(torch.randn(8, 3), dim=-1)
        try:
            ref = ref_shim.build_reference(to_plain(cfg), P.DS)
            with torch.no_grad():
                render_chunked(rays, ref, {}, 8)
            failures[name] = None
        except Exception as e:  # noqa: BLE001 - the record is the exception itself
            failures[name] = [type(e).__name__, str(e)[:200]]
    meta["reference_fails"] = failures

    # regulariser terms and re-sampled tables of the grid up-sampling step
    regularizers_package()
    from nlf.regularizers.tensorf import TVLoss as RefTV
    for name in P.UPSAMPLE_YAMLS:
        cfg = hb.to_cfg(copy.deepcopy(yamls[name]))
        cfg.color.net.N_voxel_init, cfg.color.net.N_voxel_final = 12 ** 3, 20 ** 3
        sig = hb.lower(cfg, P.DS)
        sd = seeded_state_dict(sig, seed=4)
        ref = ref_shim.build_reference(to_plain(cfg), P.DS)
        ref.load_state_dict(sd, strict=False)
        rnet = ref.model.color_model.net
        k = f"upsample/{name}/"
        arrays[k + "terms"] = np.array([float(rnet.density_L1()), float(rnet.TV_loss_density(RefTV())),
                                        float(rnet.TV_loss_app(RefTV()))], dtype=np.float64)
        arrays[k + "n_voxel_list"] = np.array([int(v) for v in rnet.N_voxel_list], dtype=np.int64)
        reso = hb.state.n_to_reso(int(rnet.N_voxel_list[0]), torch.tensor(cfg.color.net.aabb))
        rnet.upsample_volume_grid(reso)
        arrays[k + "grid"] = np.array(rnet.gridSize.tolist(), dtype=np.int64)
        for t, v in rnet.state_dict().items():
            if any(s in t for s in ("plane", "line")):
                put_sampled(k + "table/" + t, v)

    # the TensoRF regulariser's loss over iterations
    from nlf.regularizers.tensorf import TensoRF as RefReg

    class Base(torch.nn.Module):  # what BaseRegularizer provides to this class: the system handle and the iteration counter
        def __init__(self, system, cfg):
            super().__init__()
            self._system, self.cur_iter = [system], 0

        def get_system(self):
            return self._system[0]

        def set_iter(self, i):
            self.cur_iter = i

    RefReg.__bases__ = (Base,)
    cfg = hb.to_cfg(copy.deepcopy(yamls["technicolor_z_plane"]))
    cfg.color.net.N_voxel_init = cfg.color.net.N_voxel_final = 14 ** 3
    sig = hb.lower(cfg, P.DS)
    sd = seeded_state_dict(sig, seed=6)
    ref = ref_shim.build_reference(to_plain(cfg), P.DS)
    ref.load_state_dict(sd, strict=False)
    theirs = RefReg(SimpleNamespace(is_subdivided=False, render_fn=ref), ref_shim.to_attr(P.REGULARISER_CFG))
    losses = []
    for it in range(P.REGULARISER_CALLS):
        theirs.set_iter(it)
        losses.append(float(theirs._loss(None, None, 0)))
    arrays["regulariser/loss"] = np.array(losses, dtype=np.float64)
    arrays["regulariser/tv_weight_density"] = np.array(float(theirs.TV_weight_density), dtype=np.float64)

    # sample points / distances / rgb of the round-2 families
    for name in P.STAGE_YAMLS:
        cfg = hb.to_cfg(copy.deepcopy(yamls[name]))
        cfg.color.net.N_voxel_init = cfg.color.net.N_voxel_final = 16 ** 3
        sig = hb.lower(cfg, P.DS_R2)
        sd = seeded_state_dict(sig, seed=5, density_gain=30.0)
        rays = hb.rays.for_signature(sig, 40, seed=3)
        ref = ref_shim.build_reference(to_plain(cfg), P.DS_R2)
        ref.load_state_dict(sd, strict=False)
        out = ref_shim.run_reference(ref, rays.clone(), capture=True)
        n = rays.shape[0]
        arrays[f"stages/{name}/rgb"] = f32(out["rgb"].reshape(n, 3))
        put_sampled(f"stages/{name}/points", out["_embed"]["points"].reshape(n, -1))
        put_sampled(f"stages/{name}/distances", out["_embed"]["distances"].reshape(n, -1))

    # occupancy pruning: dense alpha, mask, box, cropped tables, corrected aabb, second update
    for name, gain in P.ALPHA_CASES:
        cfg = hb.to_cfg(copy.deepcopy(yamls[name]))
        cfg.color.net.N_voxel_init = cfg.color.net.N_voxel_final = 13 ** 3
        sig = hb.lower(cfg, P.DS_ALPHA)
        sd = P.corner_occupancy(seeded_state_dict(sig, seed=8), gain)
        ref = ref_shim.build_reference(to_plain(cfg), P.DS_ALPHA)
        ref.load_state_dict(sd, strict=False)
        rnet = ref.model.color_model.net
        k = f"alpha/{name}/"
        reso = tuple(rnet.gridSize.tolist())
        arrays[k + "grid0"] = np.array(reso, dtype=np.int64)
        with torch.no_grad():
            arrays[k + "dense_alpha"] = f32(rnet.getDenseAlpha(reso)[0])
        box = rnet.updateAlphaMask(reso)
        arrays[k + "box"] = exact(box)
        arrays[k + "alpha_volume"] = exact(rnet.alphaMask.alpha_volume)
        rnet.shrink(box)
        arrays[k + "grid"] = np.array(rnet.gridSize.tolist(), dtype=np.int64)
        arrays[k + "aabb"] = exact(rnet.aabb)
        for t, v in rnet.state_dict().items():
            if any(s in t for s in ("plane", "line")):
                put_sampled(k + "table/" + t, v)
        arrays[k + "box2"] = exact(rnet.updateAlphaMask(tuple(rnet.gridSize.tolist())))

    # constants the reference's constructors build, per shipped YAML and set of dataset facts
    consts = []
    for name, plain in yamls.items():
        if plain is None:
            continue
        cfg = hb.to_cfg(copy.deepcopy(plain))
        cfg.color.net.N_voxel_init = cfg.color.net.N_voxel_final = 12 ** 3
        for fi, ds in enumerate(P.FACTS):
            try:
                hb.lower(cfg, ds)
            except UnsupportedPipeline:
                continue
            ref = ref_shim.build_reference(to_plain(cfg), ds)
            embs = ref.model.embedding_model.embeddings
            keys = list(to_plain(cfg)["embedding"]["embeddings"].keys())
            isects = [embs[i].intersect_fn for i, kk in enumerate(keys) if cfg.embedding.embeddings[kk].type == "ray_intersect"]
            it, it0 = isects[-1], isects[0]
            net = ref.model.color_model.net
            rec = {"name": name, "facts": fi, "samples": it.samples.reshape(-1).float().tolist(),
                   "z_scale": torch.as_tensor(it.z_scale).reshape(-1).float().tolist(),
                   "masked": bool(it.cur_iter <= it.mask_stop_iters),
                   "distance_scale": float(net.distance_scale), "weight_thre": float(net.rayMarch_weight_thres),
                   "white_bg": bool(net.white_bg), "black_bg": bool(net.black_bg),
                   "aabb": [float(v) for v in net.aabb.reshape(-1)], "grid": net.gridSize.tolist()}
            if len(isects) > 1:  # cascade: the first, coarse intersection
                rec["pre_samples"] = it0.samples.reshape(-1).float().tolist()
                rec["pre_z_scale"] = float(torch.as_tensor(it0.z_scale).reshape(-1)[0])
            if rec["masked"]:  # otherwise nothing is masked and the bounds are irrelevant
                rec["near"], rec["far"] = float(it.near), float(it.far)
            cf = getattr(it, "contract_fn", None)
            if cf is not None and hasattr(cf, "contract_start_radius"):
                rec["contract"] = [float(cf.contract_start_radius), float(cf.contract_end_radius),
                                   float(cf.contract_start_distance), float(cf.contract_end_distance)]
            if hasattr(net, "num_keyframes"):
                rec["frames"] = [int(net.num_keyframes), int(net.total_num_frames)]
            consts.append(rec)
    meta["constants"] = consts

    # every activation module of every shipped YAML that lowers, at render iteration
    acts = {}
    for name, plain in yamls.items():
        if plain is None:
            continue
        cfg = hb.to_cfg(copy.deepcopy(plain))
        try:
            hb.lower(cfg, P.DS_R2)
        except UnsupportedPipeline:
            continue
        for _, acfg in P.walk_activations(epochs_to_iters(to_plain(cfg), 1)["embedding"]):
            if isinstance(acfg, dict) and "type" not in acfg:
                continue
            key = P.activation_key(acfg)
            if key in acts:
                continue
            mod = get_activation(ref_shim.to_attr(copy.deepcopy(acfg)) if isinstance(acfg, dict) else acfg)
            if hasattr(mod, "set_iter"):
                mod.set_iter(RENDER_ITER)
            acts[key] = mod(P.activation_inputs()).tolist()
    meta["activations"] = acts

    arrays["meta_json"] = np.frombuffer(json.dumps(meta).encode(), dtype=np.uint8)  # utf-8: a quarter of numpy's str
    np.savez_compressed(OUT, **arrays)
    print(OUT, os.path.getsize(OUT), "bytes,", len(arrays), "arrays")


if __name__ == "__main__":
    main()
