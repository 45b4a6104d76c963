"""Regenerates the golden data taken from the reference project (JokerJohn/Cloud_Map_Evaluation), unmodified:

    python tests/golden/make_golden.py <path to a checkout of the reference project>

Data fixtures of the reference, not source code:
  map_eval/scripts/voxel_errors.txt         27 columns written by MapEval::calculateVMD (map_eval.cpp:292-302):
      vmin[3] vmax[3] mu_est[3] W n_gt n_est sigma_est[6: 00 01 02 11 12 22] mu_gt[3] sigma_gt[6]
  map_eval/scripts/voxel_wasserstein_cdf.txt  sorted W + (i+1)/n (map_eval.cpp:337-340)
      both stored byte for byte, xz-compressed (voxel_errors.txt is 1.7 MB as text)
  map_eval/config/config*.yaml              the shipped MapEval configs, copied to reference_config/
Known answers of the same run, from the README run log (README.md:170, image-20250214100110872.png):
  VMD 0.35303, SCS 0.78121 (printed with setprecision(5), map_eval.cpp:462-463).
"""
import json
import lzma
import os
import shutil
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
CONFIGS = ("config.yaml", "config_building_day.yaml", "config_corridor.yaml", "config_geode.yaml")


def main(ref):
    scripts = os.path.join(ref, "map_eval", "scripts")
    for name in ("voxel_errors.txt", "voxel_wasserstein_cdf.txt"):
        with open(os.path.join(scripts, name), "rb") as f:
            raw = f.read()
        with lzma.open(os.path.join(HERE, name + ".xz"), "wb", preset=9 | lzma.PRESET_EXTREME) as f:
            f.write(raw)
    rows = np.loadtxt(lzma.open(os.path.join(HERE, "voxel_errors.txt.xz"), "rt"))
    cdf = np.loadtxt(lzma.open(os.path.join(HERE, "voxel_wasserstein_cdf.txt.xz"), "rt"))
    assert rows.shape == (7129, 27) and cdf.shape == (7129, 2)
    os.makedirs(os.path.join(HERE, "reference_config"), exist_ok=True)
    for name in CONFIGS:
        shutil.copyfile(os.path.join(ref, "map_eval", "config", name), os.path.join(HERE, "reference_config", name))
    with open(os.path.join(HERE, "readme_run_log.json"), "w") as f:
        json.dump({"source": "README.md:170 (image-20250214100110872.png), scene redbird_02",
                   "voxel_size": 3.0, "VMD": 0.35303, "SCS": 0.78121, "print_precision": 5,
                   "n_est": 12795056, "n_gt": 132012045}, f, indent=1)
    print("rows", rows.shape, "cdf", cdf.shape, os.path.getsize(os.path.join(HERE, "voxel_errors.txt.xz")), "bytes")


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit(__doc__)
    main(sys.argv[1])
