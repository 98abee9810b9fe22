"""Worker for tests/test_kd_build_paths.py: builds kd trees with the NAV_KD_MIDCAP this process was started with (the
library reads the variable once) and exports them.

usage: kd_build_worker.py IN.npz OUT.npz
IN holds kind / n / split arrays naming the point sets of test_kd_build_paths.family(); OUT gets nodes_<i>, oidx_<i>,
axes_<i> (KdTree.export(with_axes=True), built from the host through nav_kdtree_build_ex) and launches_<i>."""
import importlib
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)


def main(src, dst):
    pkg = importlib.import_module("nav-slam_b200")
    from test_kd_build_paths import family
    data = np.load(src)
    out = {}
    for i, (kind, n, split) in enumerate(zip(data["kind"], data["n"], data["split"])):
        tree = pkg.KdTree(family(str(kind), int(n)), device=0, split=str(split))
        try:
            out[f"nodes_{i}"], out[f"oidx_{i}"], out[f"axes_{i}"] = tree.export(with_axes=True)
            out[f"launches_{i}"] = np.array(tree.launch_count())
        finally:
            tree.close()
    np.savez(dst, **out)


if __name__ == "__main__":
    main(sys.argv[1], sys.argv[2])
