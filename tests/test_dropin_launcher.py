"""Drop-in tests of the host-side mirror: dataset classes against the reference's collect_pc goldens and the synthetic
dataset tree."""
import os

import numpy as np


def test_dataset_crop_matches_reference_golden(golden_dir):
    from pointnetgpd_b200.model.dataset import crop_points
    g = np.load(os.path.join(golden_dir, "collect_pc.npz"))
    for i in range(len(g["grasps"])):
        idx, pts = crop_points(g["grasps"][i], g["pc"], g["transform"])
        assert np.array_equal(idx, g[f"in_ind_{i}"])
        if len(idx):
            assert np.abs(pts - g[f"pc_t_{i}"]).max() < 1e-12


def test_synthetic_tree_and_dataset_contract(tmp_path, monkeypatch):
    from pointnetgpd_b200.synth import make_tree
    root = make_tree(str(tmp_path / "data"), train_rows=40, test_rows=10, views=2, points=6000)
    monkeypatch.setenv("PointNetGPD_FOLDER", root)
    from pointnetgpd_b200.model.dataset import PointGraspOneViewDataset, PointGraspMultiClassDataset
    ds = PointGraspOneViewDataset(grasp_points_num=750, grasp_amount_per_file=40, thresh_good=0.6, thresh_bad=0.6,
                                  tag="train", with_obj=True)
    assert len(ds) == 40
    np.random.seed(0)
    items = [ds[i] for i in range(40)]
    kept = [it for it in items if it is not None]
    assert len(kept) >= 30
    for pts, label, name in kept:
        assert pts.shape == (3, 750) and pts.dtype == np.float64 and label in (0, 1) and name == "003_cracker_box"
        assert np.abs(pts[0]).max() < 0.085 / 4 and np.abs(pts[1]).max() < 0.085 / 2      # inside the gripper box
    labels = {l for _, l, _ in kept}
    assert labels == {0, 1}
    mc = PointGraspMultiClassDataset(obj_points_num=5000, grasp_points_num=1000, pc_file_used_num=2,
                                     grasp_amount_per_file=40, thresh_good=0.6, thresh_bad=0.6, tag="train")
    it = mc[3]
    assert it is not None and it[0].shape == (3, 1000) and it[1] in (0, 1, 2)

