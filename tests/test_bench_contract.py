"""bench.py's reference arm runs on CPU: check the JSON contract of the line it prints (one line on stdout, the keys the
driver reads).  The CUDA arm prints the same keys plus roofline / clocks / stage times (checked on the GPU box)."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--config", "C1", "--steps", "1",
                          "--warmup", "0"], capture_output=True, text=True, cwd=ROOT, timeout=600)
    assert out.returncode == 0, out.stderr
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "Mpts/s" and d["higher_is_better"] is True
    assert d["metric"].startswith("Mpts/s full AC+CD+AWD+MME pass")
    assert d["value"] > 0 and d["ms_per_step"] > 0 and d["n_gpus"] == 1 and d["steps"] == 1
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "Mpts/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and d["data"] == "synthetic" and d["dtype"] == "f64"


def test_reference_arm_other_ranks_stay_silent():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                          "--warmup", "0"], capture_output=True, text=True, cwd=ROOT, env=env, timeout=120)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_dump_outputs_writes_one_float64_array_per_result_field(tmp_path):
    import numpy as np
    import bench
    from cloud_map_evaluation_b200 import _abi as A
    nn, est, awd = A.me_nn_result(), A.me_mme_result(), A.me_awd_result()
    nn.est_to_gt.rmse[2], nn.gt_to_est.n_inlier[4], nn.full_cd = 0.25, 2 ** 40 + 3, 1.5
    est.mme, est.n_valid = -3.5, 7
    awd.scs, awd.n_pairs = 0.75, 11
    bench._dump_outputs(str(tmp_path / "out"), {"nn": nn, "mme": [est], "awd": awd, "n_far": (4, 5)})
    got = {p.name[:-4]: np.load(p) for p in (tmp_path / "out").iterdir()}
    assert all(a.dtype == np.float64 for a in got.values())
    assert "mme_gt.mme" not in got and len(got) == 2 * 9 + 4 + 5 + 9 + 1
    np.testing.assert_array_equal(got["nn.est_to_gt.rmse"], [0, 0, 0.25, 0, 0])
    assert got["nn.gt_to_est.n_inlier"][4] == 2 ** 40 + 3 and got["nn.full_cd"] == 1.5
    assert got["mme_est.mme"] == -3.5 and got["mme_est.n_valid"] == 7
    assert got["awd.scs"] == 0.75 and got["awd.n_pairs"] == 11
    np.testing.assert_array_equal(got["n_far"], [4, 5])


@pytest.mark.gpu
def test_dump_outputs_same_arguments_same_outputs(tmp_path):
    """Two runs with the same arguments: `steps` timed steps each, and the same outputs (counts exactly, sums up to the
    order of the device's atomic fp64 additions), which are the ones the check block reports."""
    import numpy as np
    dumps = []
    for run in range(2):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--config", "C2", "--scale", "0.05", "--steps", "2",
                              "--warmup", "0", "--no-e2e", "--no-cpu-baseline", "--dump-outputs", str(tmp_path / str(run))],
                             capture_output=True, text=True, cwd=ROOT, timeout=600)
        assert out.returncode == 0, out.stderr
        d = json.loads(out.stdout)
        assert d["steps"] == 2
        dumps.append({p.name: np.load(p) for p in (tmp_path / str(run)).iterdir()})
    assert dumps[0].keys() == dumps[1].keys()
    for k in dumps[0]:
        if k[:-4].rsplit(".", 1)[-1].startswith("n_"):
            np.testing.assert_array_equal(dumps[0][k], dumps[1][k], err_msg=k)
        else:
            np.testing.assert_allclose(dumps[0][k], dumps[1][k], rtol=1e-12, atol=1e-15, err_msg=k)
    got, check = dumps[1], d["check"]       # both from the second run
    np.testing.assert_array_equal(got["nn.est_to_gt.rmse.npy"], check["AC_rmse"])
    np.testing.assert_array_equal(got["nn.est_to_gt.n_inlier.npy"], check["n_inlier"])
    assert got["nn.full_cd.npy"] == check["full_cd"] and got["awd.scs.npy"] == check["scs"]
    np.testing.assert_array_equal([got["mme_est.mme.npy"], got["mme_gt.mme.npy"]], check["mme"])
