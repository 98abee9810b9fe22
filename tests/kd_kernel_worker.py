"""Worker for tests/test_nn_extreme_coordinates.py: answers nearest-neighbour sets with the kd-tree search kernel that
NAV_KD_KERNEL selects in this process (the library reads the variable once).

usage: kd_kernel_worker.py IN.npz OUT.npz
IN holds n_cases, pts_<i> / q_<i> for every case and big_pts / big_q; OUT gets idx_<i>_<split> / dist_<i>_<split>
and big_idx_<split> / big_dist_<split> for both split rules, through nav_kdtree_build_ex + nav_kdtree_nn_batch."""
import importlib
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main(src, dst):
    pkg = importlib.import_module("nav-slam_b200")
    data = np.load(src)
    cases = [(f"_{i}", data[f"pts_{i}"], data[f"q_{i}"]) for i in range(int(data["n_cases"]))]
    cases.append(("big", data["big_pts"], data["big_q"]))
    out = {}
    for tag, pts, q in cases:
        prefix, suffix = ("big_", "") if tag == "big" else ("", tag)
        for split in ("widest", "cyclic"):
            tree = pkg.KdTree(pts, device=0, split=split)
            try:
                idx, dist, _ = tree.nn_batch(q, want_nearest=False)
            finally:
                tree.close()
            out[f"{prefix}idx{suffix}_{split}"] = idx
            out[f"{prefix}dist{suffix}_{split}"] = dist
    np.savez(dst, **out)


if __name__ == "__main__":
    main(sys.argv[1], sys.argv[2])
