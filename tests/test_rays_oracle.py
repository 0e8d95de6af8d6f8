"""Camera -> rays oracle against the reference golden vectors (CPU, no reference checkout needed)."""
import os

import numpy as np
import pytest
import torch

from oracle.rays_oracle import coords_from_camera, to8b
from tests.cases_rays import RAY_CASES

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")


@pytest.mark.parametrize("name", list(RAY_CASES))
def test_ray_oracle_matches_reference_golden(name):
    c = RAY_CASES[name]
    g = np.load(os.path.join(GOLDEN, f"rays_{name}.npz"))["rays"]
    r = coords_from_camera(c["pose"], c["K"], c["W"], c["H"], c["time"], c["cam_idx"], c["use_ndc"], c["near"]).numpy()
    assert r.shape == g.shape == (c["H"] * c["W"], 8)
    assert np.abs(r - g).max() <= 2e-6 * max(1.0, np.abs(g).max())


def test_ray_oracle_matches_live_reference():
    """The 6-channel NDC rays alone (no camera index / time columns appended): the reference's get_ray_directions_K ->
    get_rays -> get_ndc_rays_fx_fy, as recorded in the first six columns of the golden vectors."""
    c = RAY_CASES["ndc_73x41"]
    ref = torch.from_numpy(np.load(os.path.join(GOLDEN, "rays_ndc_73x41.npz"))["rays"][:, :6])
    mine = coords_from_camera(c["pose"], c["K"], c["W"], c["H"], use_ndc=True, near=c["near"], c_in=6)
    assert (mine - ref).abs().max() <= 2e-6 * float(ref.abs().max())


def test_to8b_truncates_like_reference():
    x = np.array([-0.2, 0.0, 0.5, 0.999, 1.0, 1.7, 1.0 / 255 - 1e-7, 2.0 / 255 + 1e-7], dtype=np.float32)
    assert to8b(x).tolist() == [0, 0, 127, 254, 255, 255, 0, 2]
