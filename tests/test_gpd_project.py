"""GPD image projection (BaseGraspDataset.collect_pc with projection=True, PointNetGPD/model/dataset.py:15-198): the
oracle normal estimator, the CPU dataset path (pointnetgpd_b200.projection) and the CUDA kernels (csrc/project.cuh;
on the CPU through the SIMT emulator build, on the GPU through prep.project) against tests/golden/gpd_project.npz,
which the reference's own collect_pc / project_pc / cal_projection wrote (oracle/make_golden_gpd_project.py)."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

import emu_util as E
from oracle import gpd_project_np as GP
from oracle import grasp_crop_np as OC
from oracle import gpd_torch_port as GT
from pointnetgpd_b200 import _abi as A
from pointnetgpd_b200 import prep, projection, synth
from pointnetgpd_b200.model import dataset as D

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "gpd_project.npz")
SCENES = ("cluster", "column")


def _gold():
    return np.load(GOLD)


def _grasp_keys(gd, scene):
    return [f"{scene}/g{g}" for g in range(len(gd[f"{scene}/grasps"]))]


def _check_image(img, ref, chann, tol):
    """occupancy channels exact (in the image's dtype: float64 for the dataset path, float32 for the kernels), normal
    channels within tol."""
    img = np.asarray(img)
    occ = [0, 4, 8] if chann == 12 else []
    nrm = [c for c in range(chann) if c not in occ]
    assert np.array_equal(img[occ], ref[occ].astype(img.dtype))
    assert np.abs(img[nrm].astype(np.float64) - ref[nrm]).max() <= tol


def test_golden_covers_the_edge_cases():
    gd = _gold()
    # a voxel with more than 50 points: grasp 0 of the cluster scene has 80 points in one voxel, so its occupancy max is 50
    assert gd["cluster/g0/img12"][0].max() == 1.0 and (gd["cluster/g0/img12"][0] == 1.0).sum() == 1
    # a degenerate box: the column's [0,1,2] image is all zeros, the two other orders are not
    img = gd["column/g0/img12"]
    assert not img[0:4].any() and img[4:8].any() and img[8:12].any()
    assert not gd["cluster/g5/valid"] and gd["cluster/g1/valid"]


def test_oracle_matches_golden():
    gd = _gold()
    for scene in SCENES:
        pc, grasps, T = gd[f"{scene}/pc"], gd[f"{scene}/grasps"], gd[f"{scene}/transform"]
        for g, key in enumerate(_grasp_keys(gd, scene)):
            in_ind, pc_in = OC.crop(pc, grasps[g], T)
            assert np.array_equal(in_ind, gd[key + "/in_ind"]), key
            if gd[key + "/valid"]:
                center, M, _w = OC.grasp_frame(grasps[g], T)
                pc_t = (M.dot((np.asarray(pc) - center).T)).T
                nrm = GP.get_normal(pc_t, only=in_ind)[in_ind]
                assert np.array_equal(nrm, gd[key + "/normals"]), key


def test_cpu_path_matches_golden():
    gd = _gold()
    for scene in SCENES:
        pc, grasps, T = gd[f"{scene}/pc"], gd[f"{scene}/grasps"], gd[f"{scene}/transform"]
        for g, key in enumerate(_grasp_keys(gd, scene)):
            center, rows, width = D.grasp_frame(grasps[g], T)
            for chann in (3, 12):
                in_ind, img = projection.project_grasp(pc, center, rows, width, chann)
                assert np.array_equal(in_ind, gd[key + "/in_ind"]), key
                assert (img is not None) == bool(gd[key + "/valid"]), key
                if img is None:
                    continue
                assert img.shape == (chann, 60, 60) and img.dtype == np.float64
                _check_image(img, gd[key + f"/img{chann}"], chann, 1e-6)
            if gd[key + "/valid"]:
                pc_t = (np.asarray(pc) - center) @ rows.T
                nrm = projection.estimate_normals(pc, pc_t, in_ind)
                assert np.abs(nrm - gd[key + "/normals"]).max() <= 1e-6, key


def test_solver_vectorised_equals_scalar():
    """The vectorised solver of the CPU path against the oracle's scalar one, on random, rank-deficient and diagonal
    matrices (every branch of the solver)."""
    rng = np.random.RandomState(0)
    mats = []
    for _ in range(300):
        a = rng.normal(size=(3, 3))
        mats.append(a @ a.T)
    for _ in range(100):
        v = rng.normal(size=(3, 2))
        mats.append(v @ v.T)                                          # rank 2: plane
    mats += [np.diag(rng.uniform(0, 1, 3)) for _ in range(20)] + [np.diag([1.0, 1.0, 2.0]), np.zeros((3, 3))]
    mats.append(np.outer([1.0, 2.0, 3.0], [1.0, 2.0, 3.0]))          # rank 1: line
    cov = np.array([[m[0, 0], m[0, 1], m[0, 2], m[1, 1], m[1, 2], m[2, 2]] for m in mats])
    got = projection.smallest_eigenvectors(cov)
    assert got[-3].tolist() == [0.0, 0.0, 1.0] and got[-2].tolist() == [0.0, 0.0, 0.0]   # diagonal tie -> z; zero matrix -> 0
    for m, v in zip(mats, got):
        ref = GP.smallest_eigenvector([list(map(float, r)) for r in m])
        assert np.abs(v - np.array(ref)).max() <= 1e-12, (m, v, ref)
        if any(ref) and np.count_nonzero(m - np.diag(np.diag(m))):   # a unit vector of the smallest eigenvalue's eigenspace
            lam = np.linalg.eigvalsh(m)
            r = np.array(ref)
            assert abs(np.linalg.norm(r) - 1.0) < 1e-12 and abs(r @ m @ r - lam[0]) <= 1e-9 * max(abs(lam).max(), 1e-300)


@pytest.mark.parametrize("chann", [3, 12])
def test_emulated_kernels_match_golden(chann):
    lib = E.emu_lib()
    gd = _gold()
    for scene in SCENES:
        pc, grasps, T = gd[f"{scene}/pc"], gd[f"{scene}/grasps"], gd[f"{scene}/transform"]
        fr = prep.grasp_frames(grasps, T)
        offsets, _pts, idx = prep.crop(torch.tensor(pc), fr, lib=lib)
        img, valid = prep.project(torch.tensor(pc), fr, chann, lib=lib)
        img, valid = img.numpy(), valid.numpy()
        for g, key in enumerate(_grasp_keys(gd, scene)):
            assert np.array_equal(idx[int(offsets[g]):int(offsets[g + 1])].numpy(), gd[key + "/in_ind"]), key
            assert bool(valid[g]) == bool(gd[key + "/valid"]), key
            if not valid[g]:
                assert not img[g].any()
                continue
            _check_image(img[g], gd[key + f"/img{chann}"], chann, 1e-6)


def test_workspace_bytes_and_arguments():
    lib = E.emu_lib()
    small = lib.pgpd_gpd_project_workspace_bytes(1000, 4, 100, 3)
    assert 0 < small < lib.pgpd_gpd_project_workspace_bytes(1000, 4, 100, 12) < lib.pgpd_gpd_project_workspace_bytes(1000, 4, 5000, 12)
    assert lib.pgpd_gpd_project_workspace_bytes(1000, 4, 100, 6) == 0
    with pytest.raises(ValueError):
        prep.project(torch.zeros((10, 3)), prep.grasp_frames(np.zeros((1, 12)) + [0, 0, 0, 0, 1, 0, 0.08, 0, 0, 0, 0, 0]), 6,
                     lib=lib)


def _collate(batch):
    """main_1v_gpd.py's my_collate: drop the None items, then the default collate."""
    return torch.utils.data.dataloader.default_collate([b for b in batch if b is not None])


def _datasets(chann):
    one = dict(grasp_points_num=750, tag="train", grasp_amount_per_file=40, thresh_good=0.6, thresh_bad=0.6,
               projection=True, project_chann=chann, project_size=60)                                 # main_1v_gpd.py:58-66
    full = dict(obj_points_num=50000, grasp_points_num=1000, pc_file_used_num=20, tag="test", grasp_amount_per_file=40,
                thresh_good=0.6, thresh_bad=0.6, with_obj=True, projection=True, project_chann=chann,
                project_size=60)                                                                        # main_fullv_gpd.py:59-90
    return [D.PointGraspOneViewDataset(**one), D.PointGraspOneViewMultiClassDataset(**one), D.PointGraspDataset(**full),
            D.PointGraspMultiClassDataset(**full)]


@pytest.mark.parametrize("chann", [3, 12])
def test_datasets_feed_the_emulated_classifier(tmp_path, chann, monkeypatch):
    root = synth.make_tree(str(tmp_path / "tree"), train_rows=40, test_rows=40, views=3, points=8000, seed=3)
    monkeypatch.setenv("PointNetGPD_FOLDER", root)
    lib = E.emu_lib()
    sd = {k: np.ascontiguousarray(v.numpy()) for k, v in GT.make_gpd_state(5, chann).items()}
    m = A.Gpd()
    for name in A.GPD_LAYERS:
        getattr(m, name).w, getattr(m, name).b = sd[name + ".weight"].ctypes.data, sd[name + ".bias"].ctypes.data
    for ds in _datasets(chann):
        np.random.seed(0)
        item = next(x for x in (ds[i] for i in range(len(ds))) if x is not None)
        assert item[0].shape == (chann, 60, 60) and item[0].dtype == np.float64
        loader = torch.utils.data.DataLoader(ds, batch_size=4, shuffle=False, collate_fn=_collate)
        batch = next(iter(loader))
        x = np.ascontiguousarray(batch[0].float().numpy())
        B = x.shape[0]
        assert B >= 1 and batch[1].shape == (B,)
        assert np.isfinite(x).all() and np.abs(x[:, 1 if chann == 12 else 0]).max() > 0
        nbytes = lib.pgpd_gpd_workspace_bytes(B, chann, 0)
        ws = E.Guarded(nbytes)
        logp = np.full((B, 2), np.nan, np.float32)
        A.check(lib, lib.pgpd_gpd_forward(C.byref(m), x.ctypes.data, B, chann, 0, logp.ctypes.data, ws.addr, nbytes, None))
        ref = GT.gpd_forward({k: torch.tensor(v) for k, v in sd.items()}, torch.tensor(x)).numpy()
        assert np.abs(logp - ref).max() < 1e-4


# ---- on the GPU ---------------------------------------------------------------------------------------------------------
def _seeded_scene(P=8000, G=1024, seed=0):
    pc = synth.uniform(seed, (P, 3), -0.05, 0.05).astype(np.float32)
    grasps = np.zeros((G, 12))
    grasps[:, 0:3] = synth.uniform(seed + 1, (G, 3), -0.02, 0.02)
    grasps[:, 3:6] = synth.normal(seed + 2, (G, 3))
    grasps[:, 6] = synth.uniform(seed + 3, (G,), 0.05, 0.085)
    grasps[:, 7] = synth.uniform(seed + 4, (G,), -np.pi, np.pi)
    grasps[::97, 0:3] += 0.2                                                  # some empty boxes
    return pc, grasps


@pytest.mark.gpu
@pytest.mark.parametrize("chann", [3, 12])
def test_gpu_matches_golden(chann):
    gd = _gold()
    for scene in SCENES:
        pc, grasps, T = gd[f"{scene}/pc"], gd[f"{scene}/grasps"], gd[f"{scene}/transform"]
        img, valid = prep.project(torch.tensor(pc).cuda(), prep.grasp_frames(grasps, T), chann)
        assert img.shape == (len(grasps), chann, 60, 60) and img.dtype == torch.float32 and valid.dtype == torch.bool
        img, valid = img.cpu().numpy(), valid.cpu().numpy()
        for g, key in enumerate(_grasp_keys(gd, scene)):
            assert bool(valid[g]) == bool(gd[key + "/valid"]), key
            if valid[g]:
                _check_image(img[g], gd[key + f"/img{chann}"], chann, 1e-6)
            else:
                assert not img[g].any()


@pytest.mark.gpu
@pytest.mark.parametrize("chann", [3, 12])
def test_gpu_matches_cpu_path_and_is_deterministic(chann):
    pc, grasps = _seeded_scene()
    fr = prep.grasp_frames(grasps)
    pcd = torch.tensor(pc).cuda()
    img, valid = prep.project(pcd, fr, chann)
    img2, valid2 = prep.project(pcd, fr, chann)
    assert torch.equal(img, img2) and torch.equal(valid, valid2)               # bit-identical from run to run
    img, valid = img.cpu().numpy(), valid.cpu().numpy()
    assert 0 < valid.sum() < len(grasps)
    from scipy.spatial import cKDTree
    tree = cKDTree(pc.astype(np.float64))
    occ = [0, 4, 8] if chann == 12 else []
    nrm = [c for c in range(chann) if c not in occ]
    for g in range(len(grasps)):
        center, rows, width = D.grasp_frame(grasps[g], np.eye(4))
        _in, ref = projection.project_grasp(pc, center, rows, width, chann, tree=tree)
        assert bool(valid[g]) == (ref is not None), g
        if ref is None:
            assert not img[g].any()
            continue
        assert np.array_equal(img[g][occ], ref[occ].astype(np.float32)), g                 # occupancy and voxel choice
        assert np.abs(img[g][nrm] - ref[nrm]).max() <= 1e-5, g


@pytest.mark.gpu
def test_gpu_loader_trains_the_cuda_classifier(tmp_path, monkeypatch):
    """main_1v_gpd.py's shape of use: the projection dataset through a None-dropping DataLoader into the CUDA
    GPDClassifier for a few SGD steps on one fixed batch; the loss is finite and decreases."""
    from pointnetgpd_b200.model.gpd import GPDClassifier
    root = synth.make_tree(str(tmp_path / "tree"), train_rows=64, test_rows=8, views=2, points=8000, seed=5)
    monkeypatch.setenv("PointNetGPD_FOLDER", root)
    ds = D.PointGraspOneViewDataset(grasp_points_num=750, tag="train", grasp_amount_per_file=64, thresh_good=0.6,
                                    thresh_bad=0.6, projection=True, project_chann=12, project_size=60)
    np.random.seed(1)
    loader = torch.utils.data.DataLoader(ds, batch_size=32, shuffle=False, collate_fn=_collate)
    data, target = next(iter(loader))
    data, target = data.float().cuda(), target.cuda()
    torch.manual_seed(0)
    m = GPDClassifier(12).cuda().train()
    opt = torch.optim.SGD(m.parameters(), lr=0.01)
    losses = []
    for _ in range(5):
        opt.zero_grad()
        loss = torch.nn.functional.nll_loss(m(data), target)
        loss.backward()
        opt.step()
        losses.append(float(loss))
    assert np.isfinite(losses).all() and losses[-1] < losses[0], losses
