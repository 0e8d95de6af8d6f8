"""Host-side logic that needs no GPU: config lowering, registry surface, chunk loop, state_dict layout,
C-ABI symbol table."""
import copy
import os
import re

import pytest
import torch

import hyperreel_b200 as hb
from hyperreel_b200 import lib as L
from hyperreel_b200.signature import UnsupportedPipeline, lower
from hyperreel_b200.state import n_to_reso, seeded_state_dict
from tests import reference_pins

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_c_abi_library_loads_and_exports_every_declared_symbol():
    header = open(os.path.join(ROOT, "include", "hyperreel_b200.h")).read()
    declared = set(re.findall(r"\b(hr_[a-z0-9_]+)\s*\(", header))
    assert declared == set(L.EXPORTS), declared ^ set(L.EXPORTS)
    lib = L.load_library()
    for name in declared:
        assert getattr(lib, name) is not None
    assert lib.hr_abi_version() == L.HR_ABI_VERSION
    m = re.search(r"#define HR_ABI_VERSION (\d+)", header)
    assert int(m.group(1)) == L.HR_ABI_VERSION


def test_ctypes_struct_matches_header_field_order():
    header = open(os.path.join(ROOT, "include", "hyperreel_b200.h")).read()
    body = header[header.index("typedef struct hr_config {"):header.index("} hr_config;")]
    fields = []
    for line in body.splitlines()[1:]:
        line = line.split("/*")[0].strip()
        if not line or line.startswith("*") or line.startswith("//"):
            continue
        decl = line.rstrip(";")
        names = decl.split(None, 1)[1] if " " in decl else ""
        for n in names.split(","):
            n = re.sub(r"\[.*\]", "", n).strip()
            if n:
                fields.append(n)
    assert fields == [f[0] for f in L.hr_config._fields_]


def test_camera_struct_matches_header_field_order():
    header = open(os.path.join(ROOT, "include", "hyperreel_b200.h")).read()
    body = header[header.index("typedef struct hr_camera {"):header.index("} hr_camera;")]
    fields = []
    for line in body.splitlines()[1:]:
        line = line.split("/*")[0].strip()
        if not line:
            continue
        decl = line.rstrip(";")
        for n in decl.split(None, 1)[1].split(","):
            n = re.sub(r"\[.*\]", "", n).strip()
            if n:
                fields.append(n)
    assert fields == [f[0] for f in L.hr_camera._fields_]
    cam = hb.Camera(pose=[[1, 0, 0, 0.5], [0, 1, 0, -1], [0, 0, 1, 2]], K=[[100, 0, 32], [0, 90, 24], [0, 0, 1]], width=64,
                    height=48, time=0.5, cam_idx=2, use_ndc=True, ndc_near=0.7).to_c()
    assert (cam.fx, cam.fy, cam.cx, cam.cy, cam.width, cam.height) == (100.0, 90.0, 32.0, 24.0, 64, 48)
    assert list(cam.c2w)[3::4] == [0.5, -1.0, 2.0] and cam.use_ndc == 1 and abs(cam.ndc_near - 0.7) < 1e-7


def test_create_without_gpu_fails_loudly():
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    cfg, ds = hb.configs.get("technicolor_z_plane", n_voxels=16 ** 3)
    model = hb.LightfieldModel(cfg, dataset=ds)
    model.eval()
    with pytest.raises(RuntimeError):
        model(torch.zeros(4, 8))  # CPU rays: no fallback
    import ctypes as C
    h = C.c_void_p()
    rc = model._lib.hr_create(C.byref(model.sig.cfg), 0, C.byref(h))
    assert rc != 0 and b"no CUDA device" in model._lib.hr_last_error()


def test_lowering_technicolor():
    cfg, ds = hb.configs.get("technicolor_z_plane")
    sig = lower(cfg, ds)
    c = sig.cfg
    assert (c.c_in, c.mlp_in, c.mlp_width, c.mlp_layers, c.mlp_skip, c.mlp_out) == (8, 9, 256, 6, 3, 480)
    assert sig.mlp_layer_shapes == [(256, 9), (256, 256), (256, 256), (256, 265), (256, 256), (480, 256)]
    assert sig.head_names == ["z_vals", "spatial_flow", "sigma", "point_sigma", "point_offset", "color_scale", "color_shift"]
    assert (c.off_z, c.off_flow, c.off_sigma, c.off_point_sigma, c.off_offset, c.off_cscale, c.off_cshift) == (0, 1, 4, 5, 6, 9, 12)
    assert c.act_sigma.kind == L.ACT_SIGMOID and c.act_sigma.shift == 4.0
    assert c.act_flow.outer_fac == 0.25 and c.flow_act.outer_fac == 0.25  # the 0.25 factor is applied twice
    assert c.act_offset.kind == L.ACT_TANH and c.act_offset.outer_fac == 0.25
    assert c.isect_act.outer_fac == 0.5 and c.isect_density_off == 4 and c.offset_density_off == 5
    assert abs(c.z_scale - 2.0 / 31.0) < 1e-6 and c.samples[0] == -1.0 and c.samples[31] == 1.0
    assert c.dynamic == 1 and c.num_keyframes == 12 and c.num_frames == 50
    assert list(c.n_sigma) == [8, 0, 0] and c.shading == L.SHADE_SH and c.app_dim == 27
    assert c.distance_scale == 16.0 and c.weight_thre == 0.0 and c.use_color_scale_shift == 1


def test_lowering_donerf_uses_dataset_bounds_and_sigma_for_offset():
    cfg, ds = hb.configs.get("donerf_sphere")
    c = lower(cfg, ds).cfg
    assert c.c_in == 6 and c.mlp_in == 18 and c.n_z == 4 and c.isect_type == L.ISECT_SPHERE
    assert c.isect_near == 0.5 and c.contract_type == L.CONTRACT_MIPNERF and c.contract_samples == 1
    assert c.contract_start_radius == 1.0 and c.contract_end_radius == 15.0
    assert c.offset_density_off == c.off_sigma  # point_offset_0 has no in_density_field -> 'sigma'
    assert c.dynamic == 0 and c.shading == L.SHADE_RGB and list(c.n_sigma) == [8, 4, 4]


def test_unsupported_pipelines_raise():
    cfg, ds = hb.configs.get("technicolor_z_plane")
    bad = hb.to_cfg(hb.config.to_plain(cfg))
    bad.embedding.embeddings.ray_intersect_0.intersect.type = "cylinder_new"
    with pytest.raises(UnsupportedPipeline):
        lower(bad, ds)
    bad = hb.to_cfg(hb.config.to_plain(cfg))
    bad.embedding.embeddings.ray_intersect_0.intersect.type = "cylinder"  # 4-channel primitive behind a 1-channel head
    with pytest.raises(UnsupportedPipeline):
        lower(bad, ds)
    bad = hb.to_cfg(hb.config.to_plain(cfg))
    bad.color.net.shadingMode = "MLP_Fea"
    with pytest.raises(UnsupportedPipeline):
        lower(bad, ds)
    bad = hb.to_cfg(hb.config.to_plain(cfg))
    bad.embedding.embeddings.ray_prediction_0.outputs.sigma.activation.window_epochs = 10 ** 9
    with pytest.raises(UnsupportedPipeline):
        lower(bad, ds, cur_iter=5, iters_per_epoch=4000)  # EaseValue still easing at iteration 5
    bad = hb.to_cfg(hb.config.to_plain(cfg))
    bad.embedding.embeddings.ray_prediction_0.params.ray.param.fn = "spherical"
    with pytest.raises(UnsupportedPipeline):
        lower(bad, ds)


def test_lowering_of_the_f3_families():
    """SURVEY 8 f3: BasicPE (column permutation), bbox / z_depth contraction, cylinder primitive, outward_facing (ignored
    by the old sphere / cylinder / z_plane classes, primitive.py:181-250,366-438), per-ray colour heads."""
    cfg, ds = hb.configs.get("technicolor_z_plane", variant="basic_pe")
    sig = lower(cfg, ds)
    assert sig.in_perm == [0, 1, 2, 3, 4, 5, 7, 6, 8]  # [t, sin2t, cos2t, sin4t, cos4t] <- BasicPE [t, sin2t, sin4t, cos2t, cos4t]
    cfg, ds = hb.configs.get("technicolor_z_plane", variant="bbox")
    c = lower(cfg, ds).cfg
    assert c.contract_type == L.CONTRACT_AFFINE and c.contract_samples == 1
    assert list(c.contract_affine_min) == [-2.0, -2.0, 0.5] and list(c.contract_affine_den) == [4.0, 4.0, -3.0]
    assert abs(c.contract_dist_fac - (4.0 + 4.0 + 3.0) / 3.0) < 1e-6
    initial = float(cfg.embedding.embeddings.ray_intersect_0.intersect.initial)
    assert abs(c.samples[0] - initial / c.contract_dist_fac) < 1e-6  # contract_distance(initial) (contract.py:80-81)
    cfg, ds = hb.configs.get("technicolor_z_plane", variant="z_depth")
    c = lower(cfg, ds).cfg
    assert c.contract_type == L.CONTRACT_AFFINE and list(c.contract_affine_den) == [1.5, 1.5, 1.5] and c.contract_dist_fac == 1.5
    cfg, ds = hb.configs.get("donerf_sphere", variant=["cylinder", "outward_facing"])
    c = lower(cfg, ds).cfg
    assert c.isect_type == L.ISECT_CYLINDER and c.n_z == 4
    cfg, ds = hb.configs.get("technicolor_z_plane", variant="global_color")
    c = lower(cfg, ds).cfg
    assert c.use_color_scale_shift == 0 and c.off_cscale_global == 9 and c.off_cshift_global == 12
    cfg, ds = hb.configs.get("technicolor_z_plane", variant="both_color")
    c = lower(cfg, ds).cfg
    assert c.use_color_scale_shift == 1 and c.off_cscale_global == 15 and c.head_stride == 21
    cfg, ds = hb.configs.get("neural_3d_z_plane", variant=["sphere", "outward_facing"])
    c = lower(cfg, ds).cfg
    assert c.isect_type == L.ISECT_SPHERE and c.dynamic == 1 and c.contract_type == L.CONTRACT_MIPNERF


def _shipped_yaml(name):
    """One of the reference's shipped model YAMLs (conf/experiment/model/<name>.yaml), from the stored record."""
    return hb.to_cfg(copy.deepcopy(reference_pins.model_yamls()[name]))


def test_shipped_model_yamls_that_lower_to_the_fused_path():
    """Coverage ledger over the reference's 51 shipped model YAMLs: these must lower (DESIGN.md section 7 lists why the
    rest are rejected)."""
    ds = {"num_keyframes": 12, "num_frames": 50, "near": 0.5, "far": 10.0, "depth_range": [0.5, 10.0], "name": "x", "collection": "y",
          "bbox_min": [-1.5, -1.25, -1.0], "bbox_max": [1.5, 1.25, 1.0], "total_images_per_frame": 5, "val_all": True}
    ok = set()
    for name in sorted(reference_pins.model_yamls()):
        try:
            lower(_shipped_yaml(name), ds)
            ok.add(name)
        except (UnsupportedPipeline, TypeError):  # bom_z_plane.yaml is an empty file
            pass
    expected = {
        "donerf_sphere", "donerf_cylinder", "donerf_cylinder_no_point", "donerf_cylinder_small", "llff_z_plane", "llff_z_plane_small",
        "neural_3d_z_plane", "neural_3d_z_plane_world", "shiny_z_plane_no_point",
        "shiny_z_plane_small", "shiny_z_plane_tiny", "spaces_z_plane", "spaces_z_plane_world", "stanford_z_plane",
        "stanford_z_plane_mem", "stanford_z_plane_small", "technicolor_z_plane", "technicolor_z_plane_ff",
        "technicolor_z_plane_mem", "technicolor_z_plane_small", "technicolor_z_plane_tiny", "technicolor_z_plane_large",
        "technicolor_z_plane_world", "immersive_sphere", "immersive_sphere_test", "immersive_cylinder", "immersive_cylinder_pe",
        "bom_cylinder", "catacaustics_z_plane", "catacaustics_cylinder", "shiny_z_plane", "stanford_llff_z_plane", "immersive_sphere_new", "bom_sphere",
        "catacaustics_distance",
        # round 2: voxel grids (axis-aligned and deformable), 96 / 128 / 256 samples per ray, the per-camera colour transform
        "catacaustics_voxel", "donerf_voxel", "shiny_z_deformable", "neural_3d_z_plane_static", "technicolor_z_plane_no_sample",
        "immersive_z_plane",
        # cascaded pipelines (point_prediction): a second net at the points of a first, coarse intersection
        "shiny_z_plane_cascaded", "shiny_z_plane_feedback", "technicolor_cascaded", "shiny_z_tensorf_cascaded",
    }
    assert len(ok) == 45  # every shipped YAML the unmodified reference itself can run (test_oracle_vs_reference.py holds the other 6; bom_z_plane.yaml is empty)
    assert expected <= ok, sorted(expected - ok)


def test_epochs_to_iters_rewrite():
    c = hb.to_cfg({"a": {"window_epochs": 3, "wait_epochs": 1, "x": {"max_freq_epoch": 2}}, "l": [{"stop_epochs": 4}]})
    hb.epochs_to_iters(c, 4000)
    assert c.a.window_iters == 12000 and c.a.wait_iters == 4000 and c.a.x.max_freq_iter == 8000 and c.l[0].stop_iters == 16000


def test_state_dict_names_follow_reference_layout():
    cfg, ds = hb.configs.get("technicolor_z_plane", n_voxels=32 ** 3)
    sig = lower(cfg, ds)
    sd = seeded_state_dict(sig, seed=0)
    assert sd["model.embedding_model.embeddings.0.net.layers.3.0.weight"].shape == (256, 265)
    assert sd["model.embedding_model.embeddings.0.net.layers.5.weight"].shape == (480, 256)
    assert sd["model.color_model.net.density_plane_space.0"].shape == (1, 8, 40, 40)
    assert sd["model.color_model.net.density_plane_space.1"].shape == (1, 0, 20, 40)
    assert sd["model.color_model.net.density_plane_time.0"].shape == (1, 8, 12, 20)
    assert sd["model.color_model.net.basis_mat.weight"].shape == (27, 8)
    assert sd["model.color_model.net.gridSize"].tolist() == [40, 40, 20]
    cfg, ds = hb.configs.get("donerf_sphere", n_voxels=32 ** 3)
    sd = seeded_state_dict(lower(cfg, ds), seed=0)
    assert sd["model.color_model.net.density_line.1"].shape == (1, 4, 32, 1)
    assert sd["model.color_model.net.app_plane.2"].shape == (1, 4, 32, 32)


def test_final_grid_sizes_match_survey():
    assert n_to_reso(512000000, torch.tensor([[-2.0, -2.0, -1.0], [2.0, 2.0, 1.0]])) == [1007, 1007, 503]
    assert n_to_reso(216000000, torch.tensor([[-2.0, -2.0, -2.0], [2.0, 2.0, 2.0]])) == [600, 600, 600]
    assert n_to_reso(262144000, torch.tensor([[-2.0, -1.5, -1.25], [2.0, 1.5, 1.25]])) == [823, 617, 514]


def test_render_chunked_is_chunk_invariant_with_any_render_fn():
    def fake(rays, **kw):
        return {"rgb": rays[:, :3] * 2.0 + 1.0, "aux": rays[:, 3:4]}
    rays = torch.randn(1000, 8)
    full = hb.render_chunked(rays, fake, {}, chunk=1 << 20)
    for chunk in (1, 7, 333, 1000, 5000):
        out = hb.render_chunked(rays, fake, {}, chunk=chunk)
        assert torch.equal(out["rgb"], full["rgb"]) and torch.equal(out["aux"], full["aux"])


def test_system_loads_shrunk_grid_checkpoint_shapes():
    """load_state_dict re-creates the tables at the checkpoint's gridSize (nlf/__init__.py:448-463)."""
    cfg, ds = hb.configs.get("donerf_sphere", n_voxels=16 ** 3)
    system = hb.INRSystem(hb.to_cfg({"model": cfg, "training": {"ray_chunk": 64}, "dataset": ds}))
    cfg2, _ = hb.configs.get("donerf_sphere", n_voxels=16 ** 3)
    sig = lower(cfg2, ds)
    sd = seeded_state_dict(sig, grid=[20, 12, 9], seed=3)
    system.load_state_dict({"state_dict": {"render_fn." + k: v for k, v in sd.items()}})
    net = system.render_fn.model.color_model.net
    assert net.gridSize.tolist() == [20, 12, 9]
    assert net.density_plane[1].shape == (1, 4, 9, 20) and net.app_line[2].shape == (1, 4, 20, 1)
    assert torch.equal(net.density_plane[0].data, sd["model.color_model.net.density_plane.0"])


def test_lowering_of_the_round_2_families():
    """Voxel grids (per-axis sample tables, interleaved), plane grids, 256 samples per ray, the per-camera colour transform and
    cascaded (point_prediction) pipelines, lowered from the reference's own YAML files."""
    ds ={"num_keyframes": 12, "num_frames": 50, "near": 0.5, "far": 10.0, "depth_range": [0.5, 10.0], "name": "x", "collection": "y",
          "bbox_min": [-1.5, -1.25, -1.0], "bbox_max": [1.5, 1.25, 1.0], "total_images_per_frame": 5, "val_all": True}
    c = lower(_shipped_yaml("donerf_voxel"), ds).cfg
    assert c.isect_type == L.ISECT_VOXEL and c.n_samples == 48 and c.isect_axes == 3 and c.n_z == 1
    # sample s = plane s // 3 of axis s % 3: first / last plane of every axis are the (contracted) dataset bounds
    assert c.samples[0] < 0 < c.samples[45] and c.samples[1] < 0 < c.samples[46] and c.samples[2] < 0 < c.samples[47]
    assert all(abs(c.z_scale3[a] - abs(c.samples[3 + a] - c.samples[a])) < 1e-6 for a in range(3))
    c = lower(_shipped_yaml("shiny_z_deformable"), ds).cfg
    assert c.isect_type == L.ISECT_PLANE and c.n_z == 4 and c.isect_axes == 1 and list(c.plane_normal)[:3] == [0.0, 0.0, 1.0]
    assert c.plane_normal_scale == 1.0
    sig = lower(_shipped_yaml("neural_3d_z_plane_static"), ds)
    assert sig.n_samples == 256 and sig.cfg.mlp_out == 256 * 14 and sig.cfg.dynamic == 0
    sig = lower(_shipped_yaml("immersive_z_plane"), ds)
    assert sig.cfg.n_color_views == 5 and sig.cfg.c_in == 8 and sig.color_views == 5 and sig.color_embedding_index > 0
    assert abs(sig.cfg.act_ctransform.inner_fac - 0.1) < 1e-7
    off = dict(ds, val_all=False)
    assert lower(_shipped_yaml("immersive_z_plane"), off).cfg.n_color_views == 0  # ColorTransformEmbedding is a no-op then
    sig = lower(_shipped_yaml("technicolor_cascaded"), ds)
    c = sig.cfg
    assert c.cascade == 1 and c.pre_samples == 8 and c.n_samples == 32 and sig.net_index == 2
    assert sig.pre_layer_shapes[-1] == (8, 256) and sig.mlp_layer_shapes[-1] == (c.mlp_out // 8, 256)
    assert list(c.pt_src) == [0, 1, 2, 3, 4, 5, 9, -1]  # points, viewdirs, times
    assert c.pre_mlp_mode == c.mlp_mode and c.pre_near == float("-inf")  # mask.stop_iters: -1 -> nothing masked
    c = lower(_shipped_yaml("shiny_z_plane_cascaded"), ds).cfg
    assert c.cascade == 1 and c.pre_mlp_mode == L.MLP_ZERO  # zero ray net: the first stage is the bare z-planes
    sd = seeded_state_dict(sig, seed=1)
    assert sd["model.embedding_model.embeddings.2.net.layers.0.0.weight"].shape == (256, 24)
    assert sd["model.embedding_model.embeddings.0.net.layers.5.weight"].shape == (8, 256)
