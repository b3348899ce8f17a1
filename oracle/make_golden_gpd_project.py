#!/usr/bin/env python
"""Generate tests/golden/gpd_project.npz by running the UNMODIFIED reference dataset code.

TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).

Run where a checkout of the reference project is available:
    python oracle/make_golden_gpd_project.py /path/to/reference-checkout
(the directory that holds PointNetGPD/).  The reference's BaseGraspDataset.collect_pc, project_pc and cal_projection
(PointNetGPD/model/dataset.py:15-198) are pulled out of the file with `ast`, as make_golden.run_collect_pc does (the module
itself needs open3d), and executed as is against a stub `self` whose get_normal is the oracle estimator
(oracle/gpd_project_np.py).  The fixture holds numbers only: per scene and grasp, in_ind, the oracle normals of the in-box
points, and the item the dataset yields for project_chann 3 and 12 (the [60,60,C] projection transposed to [C,60,60],
dataset.py:270), or valid = 0 where the item is None.  Re-running the script reproduces the file bit for bit.
"""
import ast
import os
import sys
import textwrap
import types

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
from oracle import gpd_project_np as GP  # noqa: E402
from oracle import grasp_crop_np as OC  # noqa: E402
from oracle import weights as W  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden", "gpd_project.npz")


def scenes():
    """Seeded clouds and grasps: (name, pc float32 [P,3], grasps [G,12], transform 4x4).
    `cluster`: a rotated cloud whose grasp 0 holds 80 points inside one voxel (more than voxel_point_num = 50), plus
    grasps at random poses and one whose box is empty.  `column`: every in-box point on one line along the box's z axis
    (its [0,1,2] image degenerates, dataset.py:153-157), with out-of-box points close enough that each neighbourhood
    spans three dimensions."""
    th = 0.4
    T = np.eye(4)
    T[:3, :3] = [[np.cos(th), 0, np.sin(th)], [0, 1, 0], [-np.sin(th), 0, np.cos(th)]]
    T[:3, 3] = [0.004, -0.003, 0.002]
    G = 6
    grasps = np.zeros((G, 12))
    grasps[:, 0:3] = W.uniform(301, (G, 3), -0.02, 0.02)
    grasps[:, 3:6] = W.normal(302, (G, 3))
    grasps[:, 6] = W.uniform(303, (G,), 0.06, 0.085)
    grasps[:, 7] = W.uniform(304, (G,), -1.5, 1.5)
    grasps[0, 0:8] = [0, 0, 0, 0, 1, 0, 0.08, 0]
    grasps[5, 0:3] = [0.3, 0, 0]
    center, rows, width = OC.grasp_frame(grasps[0], T)
    res = width / 59
    local = W.uniform(305, (80, 3), 0.2 * res, 0.8 * res)
    cluster = center + local @ rows
    pc_a = np.concatenate([W.uniform(306, (1200, 3), -0.05, 0.05), cluster]).astype(np.float32)
    # column: axis-aligned grasp at the origin, identity transform -> grasp-frame (x, y, z) = (x, y, -z) exactly
    col = np.zeros((60, 3))
    col[:, 0], col[:, 1], col[:, 2] = 0.019, 0.003, W.uniform(307, (60,), -0.018, 0.018)
    slab = np.stack([W.uniform(308, (3000,), 0.0205, 0.035), W.uniform(309, (3000,), -0.045, 0.045),
                     W.uniform(310, (3000,), -0.03, 0.03)], axis=1)
    pc_b = np.concatenate([slab[:1500], col, slab[1500:]]).astype(np.float32)
    g_b = np.zeros((1, 12))
    g_b[0, 0:8] = [0, 0, 0, 0, 1, 0, 0.08, 0]
    return [("cluster", pc_a, grasps, T), ("column", pc_b, g_b, np.eye(4))]


def reference_functions(ref_root):
    path = os.path.join(ref_root, "PointNetGPD", "model", "dataset.py")
    src = open(path).read()
    ns = {"np": np}
    for node in ast.walk(ast.parse(src)):
        if isinstance(node, ast.FunctionDef) and node.name in ("collect_pc", "project_pc", "cal_projection"):
            exec(textwrap.dedent(ast.get_source_segment(src, node)), ns)
    return ns


def run(ref_root):
    ns = reference_functions(ref_root)
    out = {}
    for name, pc, grasps, T in scenes():
        out[f"{name}/pc"], out[f"{name}/grasps"], out[f"{name}/transform"] = pc, grasps, T
        for chann in (3, 12):
            stub = types.SimpleNamespace(min_point_limit=50, projection=True, in_ind=None, project_size=60,
                                         projection_margin=1, voxel_point_num=50, project_chann=chann)
            normals = {}

            def get_normal(points, stub=stub, normals=normals):
                nrm = GP.get_normal(points, only=stub.in_ind)
                normals["in_box"] = nrm[stub.in_ind]
                return nrm
            stub.get_normal = get_normal
            stub.project_pc = types.MethodType(ns["project_pc"], stub)
            stub.cal_projection = types.MethodType(ns["cal_projection"], stub)
            for g in range(len(grasps)):
                normals.clear()
                res = ns["collect_pc"](stub, grasps[g], pc, T)
                key = f"{name}/g{g}"
                in_ind = np.asarray(stub.in_ind, dtype=np.int64)
                if chann == 3:
                    out[key + "/in_ind"] = in_ind
                    out[key + "/valid"] = np.array(res is not None)
                    if res is not None:
                        out[key + "/normals"] = normals["in_box"]
                else:
                    assert np.array_equal(out[key + "/in_ind"], in_ind)
                if res is not None:
                    out[key + f"/img{chann}"] = np.asarray(res, dtype=np.float64).transpose((2, 1, 0))
    np.savez_compressed(OUT, **out)
    print("wrote", OUT, {k: int(v.sum()) for k, v in out.items() if k.endswith("/valid")})


if __name__ == "__main__":
    if len(sys.argv) < 2 or not os.path.isdir(os.path.join(sys.argv[1], "PointNetGPD")):
        raise SystemExit("usage: python oracle/make_golden_gpd_project.py REFERENCE_CHECKOUT")
    run(os.path.abspath(sys.argv[1]))
