"""The oracle, the built-in configs and the host code against what the unmodified reference computes, recorded from the
reference itself by tests/golden/make_golden_reference_pins.py (tests/golden/reference_pins.npz): every check here
holds this project to the reference without needing a reference checkout."""
import copy

import pytest
import torch

from oracle.hyperreel_oracle import HyperReelOracle
from tests import reference_pins as P
from tests.cases import build_case


def _floatify(o):
    if isinstance(o, dict):
        return {k: _floatify(v) for k, v in o.items()}
    if isinstance(o, list):
        return [_floatify(v) for v in o]
    if isinstance(o, str):
        try:
            return float(o)  # PyYAML 1.1 reads `1e-3` as a string
        except ValueError:
            return o
    return o


def _key_order(o):
    if isinstance(o, dict):
        return [(k, _key_order(v)) for k, v in o.items()]
    if isinstance(o, list):
        return [_key_order(v) for v in o]
    return None


def _yaml(name):
    """A shipped model YAML of the reference, as the product reads it (hyperreel_b200.load_model_yaml)."""
    import hyperreel_b200 as hb

    return hb.to_cfg(copy.deepcopy(P.model_yamls()[name]))


def _close(want, got, tol, what=None):
    assert tuple(want.shape) == tuple(got.shape), (what, tuple(want.shape), tuple(got.shape))
    assert float((want - got).abs().max()) <= tol, what


@pytest.mark.parametrize("name", ["technicolor_z_plane", "neural_3d_z_plane", "donerf_sphere", "shiny_z_plane_tiny"])
def test_builtin_config_equals_reference_yaml(name):
    from hyperreel_b200 import configs
    from hyperreel_b200.config import to_plain
    ref = _floatify(P.model_yamls()[name])
    mine = _floatify(to_plain(configs.BUILTIN[name]()))
    assert ref == mine
    # ordered sections: embedding order, head order and param-group order are semantic
    e_ref, e_mine = ref["embedding"]["embeddings"], mine["embedding"]["embeddings"]
    assert list(e_ref) == list(e_mine)
    assert list(e_ref["ray_prediction_0"]["outputs"]) == list(e_mine["ray_prediction_0"]["outputs"])
    assert list(e_ref["ray_prediction_0"]["params"]) == list(e_mine["ray_prediction_0"]["params"])


@pytest.mark.parametrize("name", P.FRESH_CASES)
def test_oracle_matches_live_reference_on_fresh_rays(name):
    case = build_case(name, n=P.FRESH_RAYS)
    st = {}
    rgb = HyperReelOracle(case.model_cfg_plain, case.dataset, case.state_dict).render(case.rays.clone(), st)
    n = case.rays.shape[0]
    _close(P.array(f"fresh/{name}/rgb"), rgb, 2e-6)
    _close(*P.sampled(f"fresh/{name}/points", st["points"].reshape(n, -1)), 2e-6)
    _close(*P.sampled(f"fresh/{name}/distances", st["distances"].reshape(n, -1)), 2e-6)


@pytest.mark.parametrize("name", P.EDGE_CASES)
def test_oracle_matches_reference_on_crafted_edge_rays(name):
    """The rays of tests/test_edge_rays_gpu.py (plane-parallel, keyframe boundaries, far / centred origins, un-normalised
    directions): the oracle must still equal the unmodified reference there before it may judge the CUDA path."""
    from tests.test_edge_rays_gpu import craft

    case = build_case(name)
    rays = craft(case)
    a = P.array(f"edge/{name}/rgb")
    b = HyperReelOracle(case.model_cfg_plain, case.dataset, case.state_dict).render(rays.clone())
    assert torch.isfinite(a).all()
    assert float((a.reshape(b.shape) - b).abs().max()) <= 2e-6


def test_oracle_matches_reference_on_every_shipped_yaml_that_lowers():
    """Every model YAML the reference ships that the fused path accepts (45 of 52): the unmodified reference built from the
    YAML itself (grid shrunk to 24^3 for speed) rendered seeded rays with seeded parameters; the oracle must equal it.  This
    pins the oracle's reading of the real configuration files, not only of the built-ins and their variants."""
    import hyperreel_b200 as hb
    from hyperreel_b200.config import to_plain
    from hyperreel_b200.signature import UnsupportedPipeline
    from hyperreel_b200.state import seeded_state_dict

    checked, nonzero = [], 0
    for name in sorted(P.model_yamls()):
        cfg = _yaml(name)
        if cfg is None:  # bom_z_plane.yaml is empty
            continue
        cfg.color.net.N_voxel_init = P.SHIPPED_GRID
        cfg.color.net.N_voxel_final = P.SHIPPED_GRID
        try:
            sig = hb.lower(cfg, P.DS_R2)
        except UnsupportedPipeline:
            continue
        sd = seeded_state_dict(sig, seed=3, density_gain=30.0)
        rays = hb.rays.for_signature(sig, 48, seed=9)
        a = P.array(f"shipped/{name}/rgb")
        b = HyperReelOracle(to_plain(cfg), P.DS_R2, sd).render(rays.clone())
        assert float((a.reshape(b.shape) - b).abs().max()) <= 2e-6, name
        checked.append(name)
        nonzero += int(float(b.abs().max()) > 0)
    assert [k.split("/")[1] for k in P.keys("shipped/")] == checked  # every YAML the reference rendered is checked
    assert len(checked) >= 45 and nonzero >= 40


def test_six_shipped_yamls_do_not_run_in_the_reference_itself():
    """Coverage ledger honesty: catacaustics_sphere / refnerf_sphere (8 z channels into the 4-channel `sphere` primitive),
    shiny_z_tensorf (`z` is not a registered intersect type), donerf_z / shiny_z_depth (`epipolar` is not a registered embedding
    type) and blender_voxel (its ray_prediction has no `params`) fail inside the unmodified reference, so no implementation can
    be held to them; together with the empty bom_z_plane.yaml they are excluded from the denominator in DESIGN.md section 7.
    The record holds the error the reference raised for each; the fused path rejects each of them up front."""
    import hyperreel_b200 as hb
    from hyperreel_b200.signature import UnsupportedPipeline

    fails = P.meta("reference_fails")
    assert sorted(fails) == sorted(P.REFERENCE_FAILS)
    for name in P.REFERENCE_FAILS:
        assert fails[name] is not None and fails[name][0] in ("RuntimeError", "KeyError", "AttributeError", "TypeError"), name
        cfg = _yaml(name)
        cfg.color.net.N_voxel_init = cfg.color.net.N_voxel_final = 16 ** 3
        with pytest.raises(UnsupportedPipeline):
            hb.lower(cfg, P.DS)


@pytest.mark.parametrize("name", P.UPSAMPLE_YAMLS)
def test_grid_upsampling_and_regulariser_terms_match_the_reference(name):
    """The training-schedule pieces mirrored on the host (SURVEY.md 8 row f1): `upsample_volume_grid` re-samples every table
    exactly like the reference's (tensorf_base.py:1151-1188, tensorf_dynamic.py:394-441), and the TensoRF regulariser's terms
    (density_L1, TV on the space planes; nlf/regularizers/tensorf.py:14-96) agree on the same parameters."""
    import hyperreel_b200 as hb
    from hyperreel_b200.state import _Color, seeded_state_dict
    from hyperreel_b200.system import TVLoss

    cfg = _yaml(name)
    cfg.color.net.N_voxel_init, cfg.color.net.N_voxel_final = 12 ** 3, 20 ** 3
    sig = hb.lower(cfg, P.DS)
    sd = seeded_state_dict(sig, seed=4)
    k = f"upsample/{name}/"
    mine = _Color(sig, hb.state.default_grid(sig))
    mine.load_state_dict({k[len("model.color_model."):]: v for k, v in sd.items() if k.startswith("model.color_model.")}, strict=False)
    l1, tv_density, tv_app = P.array(k + "terms").tolist()
    assert abs(l1 - float(mine.net.density_L1())) <= 1e-7
    assert abs(tv_density - float(mine.net.TV_loss_density(TVLoss()))) <= 1e-9
    assert abs(tv_app - float(mine.net.TV_loss_app(TVLoss()))) <= 1e-7
    # the schedule: same voxel counts, same re-sampled tables
    assert P.array(k + "n_voxel_list").tolist() == [int(v) for v in mine.net.N_voxel_list]
    reso = hb.state.n_to_reso(int(mine.net.N_voxel_list[0]), torch.tensor(cfg.color.net.aabb))
    mine.net.upsample_volume_grid(reso)
    assert P.array(k + "grid").tolist() == mine.net.gridSize.tolist() == list(reso)
    got = mine.state_dict()
    tables = [t[len(k + "table/"):] for t in P.keys(k + "table/") if not t.endswith("#shape")]
    assert tables
    for t in tables:
        want, have = P.sampled(k + "table/" + t, got["net." + t])
        assert torch.equal(want, have), t


def test_tensorf_regulariser_loss_sequence_matches_the_reference():
    """hyperreel_b200.system.TensoRFRegularizer against nlf/regularizers/tensorf.py:35-96 (the unmodified class, its base
    replaced by a stand-in): same loss over several calls -- including the reference's running-weight bookkeeping (the TV
    weights decay per call, the density TV term is counted again inside the appearance term) and the L1 switch at the first
    alpha-mask iteration."""
    import hyperreel_b200 as hb
    from hyperreel_b200.state import _Color, seeded_state_dict
    from hyperreel_b200.system import TensoRFRegularizer

    cfg = _yaml("technicolor_z_plane")
    cfg.color.net.N_voxel_init = cfg.color.net.N_voxel_final = 14 ** 3
    sig = hb.lower(cfg, P.DS)
    sd = seeded_state_dict(sig, seed=6)
    mine = TensoRFRegularizer(dict(P.REGULARISER_CFG))
    net = _Color(sig, hb.state.default_grid(sig))
    net.load_state_dict({k[len("model.color_model."):]: v for k, v in sd.items() if k.startswith("model.color_model.")}, strict=False)
    theirs = P.array("regulariser/loss").tolist()
    assert len(theirs) == P.REGULARISER_CALLS
    for it, a in enumerate(theirs):
        mine.set_iter(it)
        b = float(mine.loss(net.net))
        assert abs(a - b) <= 1e-7 * max(1.0, abs(a)), (it, a, b)
    assert mine.L1_reg_weight == 4e-5 and abs(mine.TV_weight_density - float(P.array("regulariser/tv_weight_density"))) < 1e-12


def test_oracle_stages_match_the_reference_on_the_round_2_families():
    """Beyond rgb: the sample points and distances the oracle computes for the voxel-grid, plane-grid, colour-transform, 128 /
    256-sample and cascaded (point_prediction) YAMLs equal what the unmodified reference's `render_fn.embed` returns -- the GPU
    stage tests (tests/test_widened_gpu.py) lean on exactly these oracle stages."""
    import hyperreel_b200 as hb
    from hyperreel_b200.config import to_plain
    from hyperreel_b200.state import seeded_state_dict

    for name in P.STAGE_YAMLS:
        cfg = _yaml(name)
        cfg.color.net.N_voxel_init = cfg.color.net.N_voxel_final = 16 ** 3
        sig = hb.lower(cfg, P.DS_R2)
        sd = seeded_state_dict(sig, seed=5, density_gain=30.0)
        rays = hb.rays.for_signature(sig, 40, seed=3)
        st = {}
        rgb = HyperReelOracle(to_plain(cfg), P.DS_R2, sd).render(rays.clone(), st)
        n = rays.shape[0]
        _close(P.array(f"stages/{name}/rgb"), rgb.reshape(n, 3), 2e-6, name)
        _close(*P.sampled(f"stages/{name}/points", st["points"].reshape(n, -1)), 2e-6, name)
        _close(*P.sampled(f"stages/{name}/distances", st["distances"].reshape(n, -1)), 2e-6, name)


@pytest.mark.parametrize("name,gain", P.ALPHA_CASES)
def test_alpha_mask_update_and_shrink_match_the_reference(name, gain):
    """The pruning step of the training schedule (tensorf_base.py:379-429,1190-1232 / tensorf_dynamic.py:443-541): dense
    occupancy, mask, bounding box, cropped tables and corrected aabb equal the unmodified reference's on the same parameters;
    a second mask update (which, in the static net, consults the first mask) as well."""
    import hyperreel_b200 as hb
    from hyperreel_b200.state import _Color, seeded_state_dict

    cfg = _yaml(name)
    cfg.color.net.N_voxel_init = cfg.color.net.N_voxel_final = 13 ** 3
    sig = hb.lower(cfg, P.DS_ALPHA)
    sd = P.corner_occupancy(seeded_state_dict(sig, seed=8), gain)
    mine = _Color(sig, hb.state.default_grid(sig))
    mine.load_state_dict({k[len("model.color_model."):]: v for k, v in sd.items() if k.startswith("model.color_model.")}, strict=False)
    k = f"alpha/{name}/"
    reso = tuple(P.array(k + "grid0").tolist())
    assert reso == tuple(mine.net.gridSize.tolist())
    a_ref = P.array(k + "dense_alpha")
    with torch.no_grad():
        a_mine, _ = mine.net.getDenseAlpha(reso)
    # (the reference evaluates slab by slab, here in one batch: the same values up to the last bit or two)
    _close(a_ref, a_mine, 1e-6)
    assert float(a_ref.max()) > 0.05 > 0.001 > float(a_ref.min())
    box_ref = P.array(k + "box")
    box_mine = mine.net.updateAlphaMask(reso)
    assert torch.equal(box_ref, box_mine)
    assert torch.equal(P.array(k + "alpha_volume"), mine.net.alphaMask.volume)
    mine.net.shrink(box_mine)
    grid = P.array(k + "grid").tolist()
    assert grid == mine.net.gridSize.tolist() and any(g < r for g, r in zip(grid, reso))
    assert torch.equal(P.array(k + "aabb"), mine.net.aabb)
    got = mine.state_dict()
    tables = [t[len(k + "table/"):] for t in P.keys(k + "table/") if not t.endswith("#shape")]
    assert tables
    for t in tables:
        want, have = P.sampled(k + "table/" + t, got["net." + t])
        assert torch.equal(want, have), t
    reso2 = tuple(mine.net.gridSize.tolist())
    assert torch.equal(P.array(k + "box2"), mine.net.updateAlphaMask(reso2))


def test_lowered_constants_equal_the_reference_constructors_on_every_shipped_yaml():
    """hyperreel_b200.signature.lower (product host code) against the objects the unmodified reference builds from the same YAML
    and dataset facts: base primitives (`samples`), their spacing (`z_scale`), the mask bounds, the contraction radii, and the
    colour net's scalars -- for all 45 shipped model YAMLs that run, under two sets of dataset facts."""
    import hyperreel_b200 as hb
    from hyperreel_b200 import lib as L
    from hyperreel_b200.signature import UnsupportedPipeline

    records = {(r["name"], r["facts"]): r for r in P.meta("constants")}
    checked = 0
    for name in sorted(P.model_yamls()):
        cfg = _yaml(name)
        if cfg is None:
            continue
        cfg.color.net.N_voxel_init = cfg.color.net.N_voxel_final = 12 ** 3
        for fi, ds in enumerate(P.FACTS):
            try:
                sig = hb.lower(cfg, ds)
            except UnsupportedPipeline:
                continue
            c = sig.cfg
            rec = records[(name, fi)]
            S = c.n_samples
            assert torch.equal(torch.tensor(list(c.samples)[:S]), torch.tensor(rec["samples"])), name
            zs = torch.tensor(rec["z_scale"])
            if c.isect_type == L.ISECT_VOXEL:
                assert torch.equal(torch.tensor(list(c.z_scale3)), zs), name
            else:
                assert abs(c.z_scale - float(zs[0])) <= 1e-7 * max(1.0, abs(float(zs[0]))), name
            f32 = lambda v: float(torch.tensor(float(v), dtype=torch.float32))  # the struct holds fp32, like the tensors they meet
            if rec["masked"]:  # otherwise nothing is masked and the bounds are irrelevant
                assert c.isect_near == f32(rec["near"]) and c.isect_far == f32(rec["far"]), name
            if c.contract_type == L.CONTRACT_MIPNERF:
                r0, r1, d0, d1 = rec["contract"]
                assert (c.contract_start_radius, c.contract_end_radius) == (f32(r0), f32(r1)), name
                assert (c.contract_start_distance, c.contract_end_distance) == (f32(d0), f32(d1)), name
            if c.cascade:
                assert torch.equal(torch.tensor(list(c.pre_samples_tab)[:c.pre_samples]), torch.tensor(rec["pre_samples"])), name
                assert abs(c.pre_z_scale - rec["pre_z_scale"]) <= 1e-7, name
            assert c.distance_scale == f32(rec["distance_scale"]) and c.weight_thre == f32(rec["weight_thre"]), name
            assert bool(c.white_bg) == rec["white_bg"] and bool(c.black_bg) == rec["black_bg"], name
            assert [c.aabb[i] for i in range(6)] == [f32(v) for v in rec["aabb"]], name
            assert hb.state.default_grid(sig) == rec["grid"], name
            if c.dynamic:
                assert [c.num_keyframes, c.num_frames] == rec["frames"], name
            checked += 1
    assert checked == len(records) == 90


def test_lowered_activations_equal_the_reference_modules_on_every_shipped_yaml():
    """signature.resolve_activation lowers every head / intersect / flow / offset activation to y = f(x * inner + shift) * outer
    (the form the kernels evaluate): the same numbers as the reference's activation modules at render iteration, for every
    activation of all shipped YAMLs that lower."""
    import hyperreel_b200 as hb
    from hyperreel_b200 import lib as L
    from hyperreel_b200.config import epochs_to_iters, to_plain
    from hyperreel_b200.signature import RENDER_ITER, UnsupportedPipeline, resolve_activation

    recorded = P.meta("activations")
    x = P.activation_inputs()
    n = 0
    for name in sorted(P.model_yamls()):
        cfg = _yaml(name)
        if cfg is None:
            continue
        try:
            hb.lower(cfg, P.DS_R2)
        except UnsupportedPipeline:
            continue
        plain = epochs_to_iters(to_plain(cfg), 1)
        for path, acfg in P.walk_activations(plain["embedding"]):
            if isinstance(acfg, dict) and "type" not in acfg:
                continue
            try:
                act = resolve_activation(hb.to_cfg(acfg) if isinstance(acfg, dict) else acfg, RENDER_ITER)
            except UnsupportedPipeline:
                continue  # an activation of an embedding the fused path does not evaluate (e.g. angular flow): never lowered
            want = torch.tensor(recorded[P.activation_key(acfg)])
            v = x * act.inner_fac + act.shift
            v = torch.sigmoid(v) if act.kind == L.ACT_SIGMOID else (torch.tanh(v) if act.kind == L.ACT_TANH else v)
            got = v * act.outer_fac
            assert float((got - want).abs().max()) <= 1e-6, (name, path)
            n += 1
    assert n > 300
