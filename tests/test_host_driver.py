"""Host side of the drop-in (C++): YAML loader, cloud readers and — on the GPU — a full `map_eval` run whose
map_results.txt / voxel_errors.txt are compared with the oracle."""
import os
import struct
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXE = os.path.join(ROOT, "cloud_map_evaluation_b200", "map_eval")

CONFIG = """# a MapEval config (same keys as map_eval/config/config.yaml)
registration_methods: 2
icp_max_distance: 1.0
accuracy_level: [0.2, 0.1, 0.08, 0.05, 0.01]   # trailing comment
initial_matrix:
  - [1.0, 0.0, 0.0, 0.5]
  - [0.0, 1.0, 0.0, 0.0]
  - [0.0, 0.0, 1.0, -2]
  - [0.0, 0.0, 0.0, 1.0]
estimate_map_path: {est}
gt_map_path: "{gt}"
scene_name: unit_test
save_immediate_result: true
evaluate_mme: true
use_tbb_mme: true
evaluate_gt_mme: {gt_mme}
nn_radius: 0.1
evaluate_using_initial: {initial}
evaluate_noise_gt: false
vmd_voxel_size: 0.25
downsample_size: 0.0
use_visualization: false
enable_debug: false
"""


def _jet_u8(v):
    """open3d ColorMapJet + ColorToUint8 on an array of values."""
    def interp(x, y0, x0, y1, x1):
        return np.where(x < x0, y0, np.where(x > x1, y1, (x - x0) * (y1 - y0) / (x1 - x0) + y0))

    def base(x):
        return np.where(x <= -0.75, 0.0, np.where(x <= -0.25, interp(x, 0.0, -0.75, 1.0, -0.25),
                        np.where(x <= 0.25, 1.0, np.where(x <= 0.75, interp(x, 1.0, 0.25, 0.0, 0.75), 0.0))))
    rgb = np.stack([base(v * 2 - 1.5), base(v * 2 - 1.0), base(v * 2 - 0.5)], axis=1)
    return np.round(np.clip(rgb, 0, 1) * 255).astype(np.uint8)


def _entropy_colors(ent):
    nz = ent[ent != 0]
    max_abs, min_abs = abs(nz.min()), abs(nz.max())
    norm = (np.abs(nz) - min_abs) / (max_abs - min_abs)
    eps = 1e-1
    norm = (np.log(norm + eps) - np.log(eps)) / (np.log(1.0 + eps) - np.log(eps))
    return _jet_u8(norm)


def _read_rendered(path):
    """binary PCD with FIELDS x y z rgb -> (N x 3 float32, N x 3 uint8)"""
    raw = open(path, "rb").read()
    head, data = raw.split(b"DATA binary\n", 1)
    n = int([l for l in head.decode().splitlines() if l.startswith("POINTS")][0].split()[1])
    assert "FIELDS x y z rgb" in head.decode()
    rec = np.frombuffer(data, dtype=np.dtype([("xyz", "<f4", 3), ("rgb", "<u4")]), count=n)
    rgb = np.stack([(rec["rgb"] >> 16) & 255, (rec["rgb"] >> 8) & 255, rec["rgb"] & 255], axis=1).astype(np.uint8)
    return rec["xyz"].copy(), rgb


@pytest.fixture(scope="module")
def exe():
    if not os.path.exists(EXE):
        import __graft_entry__ as g
        g.build()
    return EXE


def _dump(exe, path):
    out = subprocess.run([exe, path, "--dump-config"], capture_output=True, text=True)
    kv = dict(line.split("=", 1) for line in out.stdout.splitlines() if "=" in line)
    return out, kv


def test_yaml_loader_matches_reference_semantics(exe, tmp_path):
    cfg = tmp_path / "c.yaml"
    cfg.write_text(CONFIG.format(est=str(tmp_path / "est"), gt=str(tmp_path / "gt.pcd"), gt_mme="false", initial="true"))
    out, kv = _dump(exe, str(cfg))
    assert out.returncode == 0, out.stderr
    assert kv["registration_methods"] == "2" and float(kv["icp_max_distance"]) == 1.0
    assert [float(x) for x in kv["accuracy_level"].split(",")] == [0.2, 0.1, 0.08, 0.05, 0.01]
    m = [float(x) for x in kv["initial_matrix"].split(",")]
    assert m[3] == 0.5 and m[11] == -2.0 and m[15] == 1.0
    assert kv["estimate_map_path"].endswith("est/")              # a trailing '/' is forced (map_eval_main.cpp:165-167)
    assert kv["result_path"].endswith("est/map_results/")
    assert kv["gt_map_path"] == str(tmp_path / "gt.pcd")          # quotes stripped
    assert kv["pcd_file_name"] == "map.pcd"                       # optional key default
    assert kv["evaluate_noised_gt"] == "0"                        # the shipped spelling `evaluate_noise_gt` is NOT read (:177)
    assert kv["evaluate_mme"] == "1" and kv["evaluate_using_initial"] == "1"


@pytest.mark.parametrize("missing", ["icp_max_distance", "enable_debug", "scene_name", "nn_radius"])
def test_yaml_loader_required_keys(exe, tmp_path, missing):
    text = "\n".join(l for l in CONFIG.format(est="a", gt="b.pcd", gt_mme="false", initial="true").splitlines()
                     if not l.startswith(missing + ":"))
    cfg = tmp_path / "c.yaml"
    cfg.write_text(text)
    out, _ = _dump(exe, str(cfg))
    assert out.returncode != 0 and "Failed to parse YAML file" in out.stderr   # map_eval_main.cpp:201-207,224-227


def test_yaml_loader_optional_accuracy_level(exe, tmp_path):
    text = "\n".join(l for l in CONFIG.format(est="a", gt="b.pcd", gt_mme="false", initial="true").splitlines()
                     if not l.startswith("accuracy_level"))
    cfg = tmp_path / "c.yaml"
    cfg.write_text(text)
    out, kv = _dump(exe, str(cfg))
    assert out.returncode == 0 and kv["accuracy_level_set"] == "0"              # optional, no default (:133-137)


def _write_pcd(path, xyz, kind, extra_field=True):
    n = len(xyz)
    fields = "x y z intensity" if extra_field else "x y z"
    hdr = (f"# .PCD v0.7\nVERSION 0.7\nFIELDS {fields}\nSIZE {'4 4 4 4' if extra_field else '4 4 4'}\n"
           f"TYPE {'F F F F' if extra_field else 'F F F'}\nCOUNT {'1 1 1 1' if extra_field else '1 1 1'}\n"
           f"WIDTH {n}\nHEIGHT 1\nVIEWPOINT 0 0 0 1 0 0 0\nPOINTS {n}\nDATA {kind}\n")
    a = xyz.astype(np.float32)
    if extra_field:
        a = np.concatenate([a, np.ones((n, 1), np.float32)], axis=1)
    with open(path, "wb") as f:
        f.write(hdr.encode())
        if kind == "ascii":
            for r in a:
                f.write((" ".join(repr(float(v)) for v in r) + "\n").encode())
        elif kind == "binary":
            f.write(a.tobytes())
        else:   # binary_compressed: SoA payload, LZF stream made of literal runs only (valid LZF)
            raw = np.ascontiguousarray(a.T).tobytes()
            comp = bytearray()
            for i in range(0, len(raw), 32):
                chunk = raw[i:i + 32]
                comp.append(len(chunk) - 1)
                comp += chunk
            f.write(struct.pack("<II", len(comp), len(raw)))
            f.write(bytes(comp))


def _write_ply(path, xyz, binary):
    n = len(xyz)
    hdr = (f"ply\nformat {'binary_little_endian' if binary else 'ascii'} 1.0\nelement vertex {n}\n"
           "property double x\nproperty double y\nproperty double z\nproperty uchar red\nend_header\n")
    with open(path, "wb") as f:
        f.write(hdr.encode())
        for r in xyz:
            if binary:
                f.write(struct.pack("<dddB", r[0], r[1], r[2], 7))
            else:
                f.write(f"{float(r[0])!r} {float(r[1])!r} {float(r[2])!r} 7\n".encode())


@pytest.mark.parametrize("kind", ["ascii", "binary", "binary_compressed", "ply_ascii", "ply_binary"])
def test_cloud_readers(exe, tmp_path, kind):
    rng = np.random.RandomState(3)
    xyz = (rng.rand(500, 3) * 100 - 50).astype(np.float32).astype(np.float64)
    xyz[7, 1] = np.nan          # removed like ReadPointCloudOption(remove_nan = true)
    xyz[9, 2] = np.inf
    if kind.startswith("ply"):
        path = str(tmp_path / "c.ply")
        _write_ply(path, xyz, kind == "ply_binary")
    else:
        path = str(tmp_path / "c.pcd")
        _write_pcd(path, xyz, kind)
    out = subprocess.run([exe, "--read-cloud", path], capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    tok = out.stdout.split()
    good = xyz[np.isfinite(xyz).all(axis=1)]
    assert int(tok[1]) == len(good) == 498
    np.testing.assert_allclose([float(t) for t in tok[3:6]], good.sum(axis=0), rtol=1e-12)


@pytest.mark.gpu
def test_map_eval_end_to_end(exe, tmp_path):
    """The re-hosted executable on a synthetic PCD pair: result lines against the oracle."""
    from cloud_map_evaluation_b200 import _abi as A
    from cloud_map_evaluation_b200 import synth
    from oracle import oracle as O
    est, gt, cfg = synth.make_pair("C2", scale=0.1)      # 100k vs 100k
    est_dir = tmp_path / "est"
    est_dir.mkdir()
    _write_pcd(str(est_dir / "map.pcd"), est, "binary")
    _write_pcd(str(tmp_path / "gt.pcd"), gt, "binary_compressed", extra_field=False)
    cfgp = tmp_path / "config.yaml"
    text = CONFIG.format(est=str(est_dir), gt=str(tmp_path / "gt.pcd"), gt_mme="true", initial="true")
    text = text.replace("[1.0, 0.0, 0.0, 0.5]", "[1.0, 0.0, 0.0, 0.0]").replace("[0.0, 0.0, 1.0, -2]", "[0.0, 0.0, 1.0, 0.0]")
    cfgp.write_text(text)
    out = subprocess.run([exe, str(cfgp)], capture_output=True, text=True)
    assert out.returncode == 0, out.stdout + out.stderr
    res = (est_dir / "map_results" / "map_results.txt").read_text().splitlines()
    line = {l.split(":")[0]: l.split(":", 1)[1].split() for l in res if ":" in l}
    assert res[0].startswith("unit_test ===================== ")
    assert line["Estimated-Ground Truth point count"] == [str(len(est)), "/", str(len(gt))]
    p = A.make_nn_params([0.2, 0.1, 0.08, 0.05, 0.01], 1.0)
    onn = O.eval_nn(est, gt, p)
    np.testing.assert_allclose([float(x) for x in line["RMSE/AC"]], list(onn.est_to_gt.rmse), rtol=1e-9, atol=1e-15)
    np.testing.assert_allclose([float(x) for x in line["Comp"]], list(onn.est_to_gt.fitness), rtol=1e-12)
    assert float(line["FULL CD"][0]) == 0.0                      # path A never computes it (map_eval.h:334)
    me, mg = O.eval_mme(est, 0.1, 10), O.eval_mme(gt, 0.1, 5)
    np.testing.assert_allclose([float(x) for x in line["MME"]],
                               [me.mme, mg.mme, mg.min_abs_entropy, mg.max_abs_entropy], atol=6e-6)
    oawd, orows = O.eval_awd(est, gt, 0.25, 100, 5, want_rows=True)
    assert abs(float(line["VMD"][0]) - oawd.awd) < 6e-6 and abs(float(line["SCS"][0]) - oawd.scs) < 6e-6
    for key in ("Time load-MME-mesh-ICP-Metric-AC-FCD", "VMD Time voxelization-WD-CDF-SCS", "AC+MME Time", "CD+MME Time",
                "AWD+SCS Time"):
        assert key in line
    rows = np.loadtxt(str(est_dir / "map_results" / "voxel_errors.txt"))
    assert rows.shape == (oawd.n_pairs, 27)
    cdf = np.loadtxt(str(est_dir / "map_results" / "voxel_wasserstein_cdf.txt"))
    np.testing.assert_allclose(cdf[:, 0], np.sort(orows[:, 9]), rtol=1e-5)
    np.testing.assert_allclose(cdf[:, 1], (np.arange(len(cdf)) + 1) / len(cdf), rtol=1e-5)
    assert "INFO: Spatial Consistency Score (SCS):" in out.stdout and "MME EST-GT:" in out.stdout
    # rendered clouds (SURVEY §8f N3; map_eval.cpp:404-412, 485-499)
    res_dir = est_dir / "map_results"
    ent_pts, ent_rgb = _read_rendered(str(res_dir / "map_entropy.pcd"))
    _, oent = O.eval_mme(est, 0.1, 10, want_entropies=True)
    assert len(ent_pts) == me.n_valid
    np.testing.assert_allclose(ent_pts, est[oent != 0].astype(np.float32), rtol=0, atol=0)
    np.testing.assert_array_equal(ent_rgb, _entropy_colors(oent))
    gt_pts, _ = _read_rendered(str(res_dir / "gt_entropy.pcd"))
    assert len(gt_pts) == mg.n_valid
    raw_pts, raw_rgb = _read_rendered(str(res_dir / "raw_rendered_dis_map.pcd"))
    _, od2 = O.knn1(est, gt)
    assert len(raw_pts) == len(est)
    np.testing.assert_array_equal(raw_rgb, _jet_u8(np.minimum(od2, 0.2) / 0.2))       # squared distance vs accuracy_level[0] (quirk)
    inl_pts, inl_rgb = _read_rendered(str(res_dir / "inlier_rendered_dis_map.pcd"))
    assert len(inl_pts) == onn.est_to_gt.n_corr
    # evaluate_using_initial: false with generalized ICP (registration_methods: 2, what every shipped config sets):
    # path B = RegistrationGeneralizedICP + calculateMetrics(reg)
    cfgp.write_text(text.replace("evaluate_using_initial: true", "evaluate_using_initial: false"))
    (est_dir / "map_results" / "map_results.txt").unlink()
    out = subprocess.run([exe, str(cfgp)], capture_output=True, text=True)
    assert out.returncode == 0, out.stdout + out.stderr
    res = (est_dir / "map_results" / "map_results.txt").read_text().splitlines()
    i0 = next(i for i, l in enumerate(res) if l.startswith("Aligned cloud:"))
    Tm = np.array([[float(x) for x in res[i0].split(":", 1)[1].split()]] + [[float(x) for x in res[i0 + k].split()] for k in (1, 2, 3)])
    Tg, fit, rmse, nc, it = O.icp_generalized(est, gt, 1.0)
    np.testing.assert_allclose(Tm, Tg, atol=6e-6)                 # printed with setprecision(5)
    line = {l.split(":")[0]: l.split(":", 1)[1].split() for l in res if ":" in l}
    assert int(line["Aligned results"][1]) == nc and abs(float(line["Aligned results"][0]) - fit) < 6e-6
    pb = A.make_nn_params([0.2, 0.1, 0.08, 0.05, 0.01], 1.0, cutoff_mode=A.ME_CUTOFF_DIST_LT_R, pairing=A.ME_PAIRING_GEOMETRIC)
    ong = O.eval_nn(O.transform(est, Tg), gt, pb)
    np.testing.assert_allclose([float(x) for x in line["RMSE/AC"]], list(ong.est_to_gt.rmse), rtol=1e-6, atol=1e-12)
    # point-to-plane ICP needs normals in the ground-truth file (Open3D raises without them); an invalid method is
    # rejected before map_results.txt is touched
    (est_dir / "map_results" / "map_results.txt").unlink()
    cfgp.write_text(text.replace("evaluate_using_initial: true", "evaluate_using_initial: false")
                    .replace("registration_methods: 2", "registration_methods: 1"))
    out = subprocess.run([exe, str(cfgp)], capture_output=True, text=True)
    assert out.returncode != 0 and "requires pre-computed normal vectors" in out.stderr
    (est_dir / "map_results" / "map_results.txt").unlink()
    cfgp.write_text(text.replace("evaluate_using_initial: true", "evaluate_using_initial: false")
                    .replace("registration_methods: 2", "registration_methods: 7"))
    out = subprocess.run([exe, str(cfgp)], capture_output=True, text=True)
    assert out.returncode != 0 and "Invalid registration type" in out.stderr
    assert not (est_dir / "map_results" / "map_results.txt").exists()
    # ... point-to-point ICP (registration_methods: 0) is: path B = ICP + calculateMetrics(reg)
    cfgp.write_text(text.replace("evaluate_using_initial: true", "evaluate_using_initial: false")
                    .replace("registration_methods: 2", "registration_methods: 0"))
    out = subprocess.run([exe, str(cfgp)], capture_output=True, text=True)
    assert out.returncode == 0, out.stdout + out.stderr
    res = (est_dir / "map_results" / "map_results.txt").read_text().splitlines()
    i0 = next(i for i, l in enumerate(res) if l.startswith("Aligned cloud:"))
    Tm = np.array([[float(x) for x in res[i0].split(":", 1)[1].split()]] + [[float(x) for x in res[i0 + k].split()] for k in (1, 2, 3)])
    To, fit, rmse, nc, it = O.icp_point_to_point(est, gt, 1.0)
    np.testing.assert_allclose(Tm, To, atol=6e-6)                 # printed with setprecision(5)
    line = {l.split(":")[0]: l.split(":", 1)[1].split() for l in res if ":" in l}
    assert int(line["Aligned results"][1]) == nc and abs(float(line["Aligned results"][0]) - fit) < 6e-6
    aligned = O.transform(est, To)
    pb = A.make_nn_params([0.2, 0.1, 0.08, 0.05, 0.01], 1.0, cutoff_mode=A.ME_CUTOFF_DIST_LT_R, pairing=A.ME_PAIRING_GEOMETRIC)
    onb = O.eval_nn(aligned, gt, pb)
    np.testing.assert_allclose([float(x) for x in line["RMSE/AC"]], list(onb.est_to_gt.rmse), rtol=1e-7, atol=1e-12)
    assert abs(float(line["FULL CD"][0]) - onb.full_cd) < 6e-6     # path B computes the full Chamfer distance (:1194)


@pytest.mark.gpu
def test_map_eval_with_downsampling(exe, tmp_path):
    """downsample_size > 0 (every shipped config uses 0.01): VoxelDownSample runs on the GPU before the metric path
    (map_eval.cpp:38-39).  The down-sampled clouds come out in voxel order, so the oracle is fed the oracle's own
    down-sampling of the same input (same point set; only order-dependent quantities are excluded)."""
    from cloud_map_evaluation_b200 import _abi as A
    from cloud_map_evaluation_b200 import synth
    from oracle import oracle as O
    est, gt, cfg = synth.make_pair("C2", scale=0.1)
    est_dir = tmp_path / "est"
    est_dir.mkdir()
    _write_pcd(str(est_dir / "map.pcd"), est, "binary")
    _write_pcd(str(tmp_path / "gt.pcd"), gt, "binary")
    s = 0.03
    text = CONFIG.format(est=str(est_dir), gt=str(tmp_path / "gt.pcd"), gt_mme="false", initial="true")
    text = text.replace("[1.0, 0.0, 0.0, 0.5]", "[1.0, 0.0, 0.0, 0.0]").replace("[0.0, 0.0, 1.0, -2]", "[0.0, 0.0, 1.0, 0.0]")
    text = text.replace("downsample_size: 0.0", f"downsample_size: {s}")
    cfgp = tmp_path / "config.yaml"
    cfgp.write_text(text)
    out = subprocess.run([exe, str(cfgp)], capture_output=True, text=True)
    assert out.returncode == 0, out.stdout + out.stderr
    res = (est_dir / "map_results" / "map_results.txt").read_text().splitlines()
    line = {l.split(":")[0]: l.split(":", 1)[1].split() for l in res if ":" in l}
    de, dg = O.voxel_downsample(est, s), O.voxel_downsample(gt, s)
    assert len(de) < len(est) and len(dg) < len(gt)
    assert line["Estimated-Ground Truth point count"] == [str(len(de)), "/", str(len(dg))]
    onn = O.eval_nn(de, dg, A.make_nn_params([0.2, 0.1, 0.08, 0.05, 0.01], 1.0))
    np.testing.assert_allclose([float(x) for x in line["RMSE/AC"]], list(onn.est_to_gt.rmse), rtol=1e-9, atol=1e-15)
    np.testing.assert_allclose([float(x) for x in line["Comp"]], list(onn.est_to_gt.fitness), rtol=1e-12)
    me = O.eval_mme(de, 0.1, 10)
    assert abs(float(line["MME"][0]) - me.mme) < 6e-6
    oawd = O.eval_awd(de, dg, 0.25, 100, 5)
    assert abs(float(line["VMD"][0]) - oawd.awd) < 6e-6 and abs(float(line["SCS"][0]) - oawd.scs) < 6e-6


@pytest.mark.gpu
def test_map_eval_two_gpus_matches_one(exe, tmp_path):
    """`map_eval --gpus 2`: one context per GPU in one process, the sweeps' query ranges sharded, the accumulators
    combined with an NCCL all-reduce in the C++ driver (gpu_group.hpp).  Same result lines as the single-GPU run."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    from cloud_map_evaluation_b200 import synth
    est, gt, cfg = synth.make_pair("C2", scale=0.3)
    outs = {}
    for n in (1, 2):
        d = tmp_path / f"run{n}"
        est_dir = d / "est"
        est_dir.mkdir(parents=True)
        _write_pcd(str(est_dir / "map.pcd"), est, "binary")
        _write_pcd(str(d / "gt.pcd"), gt, "binary")
        text = CONFIG.format(est=str(est_dir), gt=str(d / "gt.pcd"), gt_mme="true", initial="true")
        text = text.replace("[1.0, 0.0, 0.0, 0.5]", "[1.0, 0.0, 0.0, 0.0]").replace("[0.0, 0.0, 1.0, -2]", "[0.0, 0.0, 1.0, 0.0]")
        text = text.replace("downsample_size: 0.0", "downsample_size: 0.02")
        (d / "config.yaml").write_text(text)
        out = subprocess.run([exe, str(d / "config.yaml"), "--gpus", str(n)], capture_output=True, text=True)
        assert out.returncode == 0, out.stdout + out.stderr
        res = (est_dir / "map_results" / "map_results.txt").read_text().splitlines()
        outs[n] = {l.split(":")[0]: l.split(":", 1)[1].split() for l in res if ":" in l and not l.startswith(("Ground", "Evaluation"))}
        if n == 2:
            assert "sharding the sweeps over 2 GPUs" in out.stdout
    for key in ("Estimated-Ground Truth point count", "Comp"):
        assert outs[1][key] == outs[2][key], key
    for key in ("RMSE/AC", "MME", "VMD", "SCS"):
        np.testing.assert_allclose([float(x) for x in outs[2][key]], [float(x) for x in outs[1][key]], rtol=1e-12, atol=1e-12, err_msg=key)
    # the rendered clouds are assembled from the per-GPU shards of the per-point results: byte-identical files
    for name in ("map_entropy.pcd", "gt_entropy.pcd", "raw_rendered_dis_map.pcd", "inlier_rendered_dis_map.pcd"):
        a = (tmp_path / "run1" / "est" / "map_results" / name).read_bytes()
        b = (tmp_path / "run2" / "est" / "map_results" / name).read_bytes()
        assert len(a) > 200 and a == b, name


@pytest.mark.parametrize("name", ["config.yaml", "config_building_day.yaml", "config_corridor.yaml", "config_geode.yaml"])
def test_loader_reads_the_references_shipped_configs(exe, golden_dir, name):
    """The YAML-subset loader on the configuration files the reference ships (map_eval/config/*.yaml), unmodified
    (copies under tests/golden/reference_config/)."""
    out, kv = _dump(exe, os.path.join(golden_dir, "reference_config", name))
    assert out.returncode == 0, out.stderr
    assert kv["registration_methods"] == "2" and float(kv["icp_max_distance"]) == 1.0
    assert [float(x) for x in kv["accuracy_level"].split(",")] == [0.2, 0.1, 0.08, 0.05, 0.01]
    assert [float(x) for x in kv["initial_matrix"].split(",")][::5] == [1.0, 1.0, 1.0, 1.0]
    assert float(kv["nn_radius"]) == 0.1 and float(kv["downsample_size"]) == 0.01
    assert kv["evaluate_using_initial"] == "0" and kv["evaluate_noised_gt"] == "0"       # `evaluate_noise_gt` is not a key the loader reads
    assert kv["estimate_map_path"].endswith("/") and kv["gt_map_path"].endswith((".pcd", ".ply"))
    assert float(kv["vmd_voxel_size"]) in (2.0, 3.0)
