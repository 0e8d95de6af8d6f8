"""bench.py helpers that need no GPU: the algorithmic byte / MAC counts behind `roofline` (SURVEY.md section 8d) and the
reference arm's JSON line."""
import json
import os
import subprocess
import sys

import hyperreel_b200 as hb

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402


def _sig(name, **over):
    cfg, ds = hb.configs.get(name, **over)
    return hb.lower(cfg, ds)


def test_algorithmic_bytes_per_ray_match_the_survey_table():
    # B_ray = 4*C_in + 12 + S * sum_fields sum_groups 4*C*(4 + T), T = 4 (time plane) or 2 (line)
    assert bench.algorithmic_bytes_per_ray(_sig("technicolor_z_plane")) == 16428
    assert bench.algorithmic_bytes_per_ray(_sig("neural_3d_z_plane")) == 65580
    assert bench.algorithmic_bytes_per_ray(_sig("donerf_sphere", z_channels=16)) == 12324
    assert bench.algorithmic_bytes_per_ray(_sig("donerf_sphere")) == 24612
    assert bench.algorithmic_bytes_per_ray(_sig("donerf_sphere", z_channels=4)) == 3108


def test_sample_net_mac_counts_match_the_survey_table():
    macs = lambda s: sum(o * i for o, i in s.mlp_layer_shapes)  # noqa: E731
    assert macs(_sig("technicolor_z_plane")) == 389632
    assert macs(_sig("donerf_sphere", z_channels=16)) == 332800
    assert macs(_sig("neural_3d_z_plane")) == 519680


def test_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` times the oracle port on the host cores (no GPU involved) and prints one JSON line."""
    env = dict(os.environ, HR_BENCH_CPU_RAYS="256")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, env=env, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "Mrays/s" and line["higher_is_better"] is True
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0
    assert line["value"] > 0 and line["config"]["workload"].startswith("technicolor_z_plane")


def test_dump_outputs_writes_the_same_rgb_on_every_run(tmp_path):
    """`--dump-outputs DIR` writes the rgb of the last timed step as DIR/rgb.npy; the inputs are seeded, so two runs with the
    same arguments write the same array (what makes two builds comparable output for output)."""
    import numpy as np

    env = dict(os.environ, HR_BENCH_CPU_RAYS="256")
    got = []
    for i in range(2):
        d = tmp_path / f"run{i}"
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                              "--dump-outputs", str(d)], capture_output=True, text=True, env=env, timeout=600)
        assert out.returncode == 0, out.stderr[-2000:]
        got.append(np.load(d / "rgb.npy"))
    assert got[0].shape == (256, 3) and got[0].dtype == np.float32 and np.isfinite(got[0]).all()
    assert np.array_equal(got[0], got[1])
