"""Pins the oracle against the only known-answer artefacts the reference ships (SURVEY.md §4):
the sample voxel_errors.txt / voxel_wasserstein_cdf.txt and the README run log of the same run."""
import json
import lzma
import os

import numpy as np

from oracle import oracle as O


def _load(golden_dir):
    rows = np.loadtxt(lzma.open(os.path.join(golden_dir, "voxel_errors.txt.xz"), "rt"))
    cdf = np.loadtxt(lzma.open(os.path.join(golden_dir, "voxel_wasserstein_cdf.txt.xz"), "rt"))
    with open(os.path.join(golden_dir, "readme_run_log.json")) as f:
        log = json.load(f)
    return rows, cdf, log


def _sym(tri):
    s = np.empty(9)
    s[[0, 1, 2, 4, 5, 8]] = tri
    s[3], s[6], s[7] = tri[1], tri[2], tri[4]
    return s


def test_wasserstein_formula_reproduces_fixture(golden_dir):
    rows, _, _ = _load(golden_dir)
    rel = []
    rel_wrong = []
    for r in rows[::3]:
        mu_e, w, n_g, n_e = r[6:9], r[9], int(r[10]), int(r[11])
        s_e, mu_g, s_g = _sym(r[12:18]), r[18:21], _sym(r[21:27])
        # reference call order (gt_voxel, est_voxel), map_eval.cpp:284
        got = O.wasserstein(mu_g, s_g, n_g, mu_e, s_e, n_e)
        rel.append(abs(got - w) / max(w, 1e-12))
        # without the third division by (n-1) (voxel_calculator.cpp:120,128) the fixture is NOT reproduced
        wrong = O.wasserstein(mu_g, s_g * (n_g - 1), n_g, mu_e, s_e * (n_e - 1), n_e)
        rel_wrong.append(abs(wrong - w) / max(w, 1e-12))
    rel, rel_wrong = np.array(rel), np.array(rel_wrong)
    # limited by the 6-significant-digit text of the fixture (mu ~ -200 m printed to 1 mm)
    assert np.median(rel) < 2e-3, np.median(rel)
    assert np.percentile(rel, 99) < 5e-2, np.percentile(rel, 99)
    assert np.median(rel_wrong) > 2 * np.median(rel)
    assert rows[:, 10].min() >= 100 and rows[:, 11].min() >= 100  # the >=100-point filter, map_eval.cpp:280


def test_cdf_file_is_sorted_w(golden_dir):
    rows, cdf, _ = _load(golden_dir)
    w = np.sort(rows[:, 9])
    np.testing.assert_allclose(cdf[:, 0], w, rtol=0, atol=0)
    n = len(w)
    np.testing.assert_allclose(cdf[:, 1], (np.arange(n) + 1) / n, rtol=1e-5)


def test_awd_and_scs_known_answers(golden_dir):
    rows, _, log = _load(golden_dir)
    v = log["voxel_size"]
    keys = np.rint(rows[:, 0:3] / v).astype(np.int32)
    assert np.abs(rows[:, 0:3] / v - keys).max() == 0
    w = rows[:, 9]
    half_ulp = 0.5 * 10 ** (-log["print_precision"])
    # 6-significant-digit inputs -> allow 2 print ulps
    assert abs(w.mean() - log["VMD"]) <= 4 * half_ulp
    scs, count = O.scs(keys, w, radius=5)
    assert abs(scs - log["SCS"]) <= 4 * half_ulp, scs
    assert count == len(w) - 1  # one voxel has no neighbour inside the 11^3 window


def test_voxel_hash_mode_changes_speed_not_results():
    """bench.py times the CPU baseline with a mixing voxel hash (the reference's XOR hash makes its voxel maps degenerate):
    counts identical, AWD / SCS equal to summation order."""
    from oracle import oracle as O
    from cloud_map_evaluation_b200 import synth
    est, gt, cfg = synth.make_pair("C2", scale=0.1)
    a = O.eval_awd(est, gt, cfg["vmd_voxel_size"], 20, 5)
    O.set_voxel_hash(True)
    try:
        b = O.eval_awd(est, gt, cfg["vmd_voxel_size"], 20, 5)
    finally:
        O.set_voxel_hash(False)
    for k in ("n_pairs", "n_scs", "n_voxels_est", "n_voxels_gt", "n_active", "n_old", "n_new"):
        assert getattr(a, k) == getattr(b, k), k
    assert a.n_pairs > 10
    np.testing.assert_allclose([a.awd, a.scs], [b.awd, b.scs], rtol=1e-12)
