"""GPU tests of the data preparation kernels (crop, resample) and of batched candidate scoring."""
import os

import numpy as np
import pytest
import torch

from golden_util import shipped_state
from oracle import grasp_crop_np as OC
from oracle import pointnet_torch_port as PT
from oracle import weights as W
from pointnetgpd_b200 import prep
from pointnetgpd_b200.model.pointnet import PointNetCls
from pointnetgpd_b200.scoring import score_candidates

pytestmark = pytest.mark.gpu


def test_crop_matches_reference_golden(golden_dir):
    g = np.load(os.path.join(golden_dir, "collect_pc.npz"))
    pc, grasps, T = g["pc"], g["grasps"], g["transform"]
    offsets, pts, idx = prep.crop(torch.tensor(pc).cuda(), prep.grasp_frames(grasps, T))
    for i in range(len(grasps)):
        a, b = int(offsets[i]), int(offsets[i + 1])
        assert np.array_equal(idx[a:b].cpu().numpy(), g[f"in_ind_{i}"]), i          # bit-exact index sets
        if b > a:
            assert np.abs(pts[a:b].cpu().numpy() - g[f"pc_t_{i}"].astype(np.float32)).max() < 1e-7


def test_crop_large_scene_vs_oracle():
    P, G = 50000, 64                                   # full-view cloud size of dataset.py:250-254, a batch of grasps
    pc = W.uniform(31, (P, 3), -0.15, 0.15).astype(np.float32)
    centers = W.uniform(32, (G, 3), -0.08, 0.08)
    grasps = np.concatenate([centers, W.normal(33, (G, 3)), W.uniform(34, (G, 1), 0.04, 0.085),
                             W.uniform(35, (G, 1), -3.0, 3.0), np.zeros((G, 4))], axis=1)
    offsets, pts, idx = prep.crop(torch.tensor(pc).cuda(), prep.grasp_frames(grasps, None))
    idx = idx.cpu().numpy()
    for i in range(G):
        ref_idx, _ = OC.crop(pc, grasps[i], np.eye(4))
        assert np.array_equal(idx[int(offsets[i]):int(offsets[i + 1])], ref_idx), i


def test_resample_gpu_properties():
    sizes = [0, 19, 20, 499, 500, 501, 3000, 20000]
    offsets = torch.tensor(np.concatenate([[0], np.cumsum(sizes)]), dtype=torch.int32)
    pts = torch.tensor(W.normal(41, (sum(sizes), 3)).astype(np.float32)).cuda()
    x, oi = prep.resample(pts, offsets, 500, repeat=4, seed=9, return_index=True)
    x2, oi2 = prep.resample(pts, offsets, 500, repeat=4, seed=9, return_index=True)
    assert torch.equal(x, x2) and torch.equal(oi, oi2)
    oi = oi.cpu().numpy()
    for c, n in enumerate(sizes):
        for r in range(4):
            ind = oi[c * 4 + r]
            if n == 0:
                assert (ind == -1).all()
                continue
            assert OC.resample_indices_ok(ind, n, 500), n
            src = pts[int(offsets[c]):int(offsets[c + 1])]
            assert torch.equal(x[c * 4 + r], src[torch.tensor(ind, device="cuda").long()].T.contiguous())


def test_score_candidates_matches_oracle(golden_dir):
    """deployment path (kinect2grasp.py:454-491) with the shipped 3-class checkpoint: batched GPU scoring vs the
    oracle evaluated on the same resampled points."""
    st = shipped_state()
    m = PointNetCls(num_points=500, k=3)
    m.load_state_dict({k: torch.tensor(v) for k, v in st.items()})
    m = m.cuda().eval()
    sizes = [5, 19, 20, 100, 499, 500, 800, 2500, 40, 1200]
    half = np.array([0.085 / 4, 0.085 / 2, 0.085 / 4])
    clouds = [(W.uniform(60 + i, (n, 3), -1, 1) * half).astype(np.float32) for i, n in enumerate(sizes)]
    pred, score = score_candidates(m, clouds, input_points_num=500, min_points=20, repeat=5, seed=123)
    assert pred.shape == (10,) and score.shape == (10,)
    assert pred[0] == 0 and score[0] == 0.0 and pred[1] == 0 and score[1] == 0.0          # < 20 points (kinect2grasp.py:462)
    # oracle: same resampling (same seed, same kernel -- checked separately), model evaluated by the torch port
    keep = [i for i, c in enumerate(clouds) if len(c) >= 20]
    offsets = torch.zeros(len(keep) + 1, dtype=torch.int32)
    offsets[1:] = torch.cumsum(torch.tensor([len(clouds[i]) for i in keep]), 0).to(torch.int32)
    cat = torch.cat([torch.tensor(clouds[i]) for i in keep], 0).cuda()
    x = prep.resample(cat, offsets, 500, repeat=5, seed=123).cpu()
    sd = PT.to_torch_state(st, torch.float32)
    with torch.no_grad():
        logp, _ = PT.pointnetcls_forward(sd, x, training=False)
    probs = logp.exp().double().numpy().reshape(len(keep), 5, 3)
    for j, i in enumerate(keep):
        v, sc = OC.vote(probs[j].argmax(1), probs[j], 2)
        assert pred[i] == v, i
        assert abs(score[i] - sc) < 1e-4, i
