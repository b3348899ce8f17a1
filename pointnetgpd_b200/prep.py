"""Host side of the data preparation in front of the model (SURVEY.md section 8f rows 1-2):
gripper-box crop of a cloud for a batch of grasps, resampling of every crop to exactly N points, and the GPD
baseline's 60 x 60 image projection of every crop -- all run in libpgpd on the GPU; this module computes the per-grasp
frames (a handful of 3x3 products per grasp) and drives the two-pass crop (count, prefix-sum, gather).

Reference semantics: BaseGraspDataset.collect_pc (PointNetGPD/model/dataset.py:15-76), the resampling of
dataset.py:438-444 / dex-net/apps/kinect2grasp.py:473-478, the projection of dataset.py:78-198.
"""
import ctypes as C

import numpy as np
import torch

from . import _abi as A


def grasp_frames(grasps, transform=None):
    """[G,15] float64 frames for pgpd_crop_box from grasp rows [G,>=8] (center3, axis3, width, angle, ...;
    dexnet ParallelJawPtGrasp3D.configuration_from_params) and the 4x4 mesh->cloud transform (dataset.py:13)."""
    g = np.asarray(grasps, dtype=np.float64)
    if g.ndim == 1:
        g = g[None]
    T = np.eye(4) if transform is None else np.asarray(transform, dtype=np.float64)
    G = g.shape[0]
    c, ax, width, ang = g[:, 0:3], g[:, 3:6], g[:, 6], g[:, 7]
    ax = ax / np.linalg.norm(ax, axis=1, keepdims=True)
    # in-plane x axis perpendicular to the closing axis; degenerate (axis along z) -> world x
    axx = np.stack([ax[:, 1], -ax[:, 0], np.zeros(G)], axis=1)
    nx = np.linalg.norm(axx, axis=1)
    axx = np.where(nx[:, None] == 0, np.array([[1.0, 0.0, 0.0]]), axx / np.where(nx == 0, 1.0, nx)[:, None])
    az = np.cross(axx, ax)
    # approach = first column of [axx ax az] * Ry(angle) = cos*axx - sin*az ... with the reference's R1 layout:
    # R1 columns are (cos,0,sin),(0,1,0),(-sin,0,cos) -> first column of R2 R1 = cos*axx + sin*az
    approach = np.cos(ang)[:, None] * axx + np.sin(ang)[:, None] * az
    approach = approach / np.linalg.norm(approach, axis=1, keepdims=True)
    minor = np.cross(ax, approach)
    R, t = T[:3, :3], T[:3, 3]
    center = c @ R.T + t
    rows = np.stack([approach @ R.T, ax @ R.T, minor @ R.T], axis=1)        # [G,3,3]
    lim = np.stack([width / 4, width / 2, width / 4], axis=1)
    return np.concatenate([center, rows.reshape(G, 9), lim], axis=1)


def _ptr(t):
    return None if t is None else t.data_ptr()


def crop(pc, frames, lib=None):
    """pc: [P,3] float32 tensor (cuda); frames: [G,15] float64.  Returns (offsets [G+1] int32 cpu, pts [total,3]
    float32, idx [total] int32): for grasp g the points inside its box are pts[offsets[g]:offsets[g+1]], ascending
    cloud index -- exactly `pc_t[in_ind]` / `in_ind` of dataset.py:51-76."""
    lib = lib or A.load()
    dev = pc.device
    pc = pc.contiguous().float()
    fr = torch.as_tensor(np.ascontiguousarray(frames), dtype=torch.float64, device=dev)
    G, P = fr.shape[0], pc.shape[0]
    stream = torch.cuda.current_stream(dev).cuda_stream if dev.type == "cuda" else None
    counts = torch.zeros(G, dtype=torch.int32, device=dev)
    A.check(lib, lib.pgpd_crop_box(_ptr(pc), P, _ptr(fr), G, None, _ptr(counts), None, None, stream))
    offsets = torch.zeros(G + 1, dtype=torch.int32)
    offsets[1:] = torch.cumsum(counts.cpu(), 0)
    total = int(offsets[-1])
    off_dev = offsets[:-1].to(dev)
    pts = torch.empty((max(total, 1), 3), dtype=torch.float32, device=dev)
    idx = torch.empty(max(total, 1), dtype=torch.int32, device=dev)
    if total > 0:
        A.check(lib, lib.pgpd_crop_box(_ptr(pc), P, _ptr(fr), G, _ptr(off_dev), None, _ptr(pts), _ptr(idx), stream))
    return offsets, pts[:total], idx[:total]


def resample(pts, offsets, N, repeat=1, seed=0, return_index=False, lib=None):
    """pts: [total,3] float32 (cuda), offsets: [C+1] int32.  Returns x [C*repeat,3,N] float32 (the model's input
    layout) and optionally the chosen indices [C*repeat,N] (relative to each set)."""
    lib = lib or A.load()
    dev = pts.device
    C_ = int(offsets.numel()) - 1
    off_dev = offsets.to(device=dev, dtype=torch.int32)
    x = torch.empty((C_ * repeat, 3, N), dtype=torch.float32, device=dev)
    oi = torch.empty((C_ * repeat, N), dtype=torch.int32, device=dev) if return_index else None
    stream = torch.cuda.current_stream(dev).cuda_stream if dev.type == "cuda" else None
    src = pts.contiguous().float() if pts.numel() else torch.zeros((1, 3), dtype=torch.float32, device=dev)
    A.check(lib, lib.pgpd_resample(_ptr(src), _ptr(off_dev), C_, N, repeat, C.c_ulonglong(seed & (2**64 - 1)),
                                   _ptr(x), _ptr(oi), stream))
    return (x, oi) if return_index else x


def project(pc, frames, chann, lib=None):
    """GPD input images of one cloud for G grasps (BaseGraspDataset.collect_pc with projection=True, dataset.py:15-198).
    pc: [P,3] float32 tensor (cuda); frames: [G,15] float64 (grasp_frames); chann: 3 or 12.  Returns (images
    [G,chann,60,60] float32 on pc's device, the layout GPDClassifier reads; valid [G] bool: the box holds >= 50 points,
    where the reference's item is None the image is all zeros).  Crop with pgpd_crop_box, then pgpd_gpd_project."""
    if chann not in (3, 12):
        raise ValueError("chann must be 3 or 12 (dataset.py:218-219)")
    lib = lib or A.load()
    dev = pc.device
    pc = pc.contiguous().float()
    offsets, _pts, idx = crop(pc, frames, lib=lib)
    fr = torch.as_tensor(np.ascontiguousarray(frames), dtype=torch.float64, device=dev)
    G, P, total = fr.shape[0], pc.shape[0], int(offsets[-1])
    nbytes = lib.pgpd_gpd_project_workspace_bytes(P, G, total, chann)
    ws = torch.empty(nbytes + 256, dtype=torch.uint8, device=dev)
    out = torch.empty((G, chann, 60, 60), dtype=torch.float32, device=dev)
    valid = torch.empty(G, dtype=torch.bool, device=dev)
    stream = torch.cuda.current_stream(dev).cuda_stream if dev.type == "cuda" else None
    idx = idx if total > 0 else torch.zeros(1, dtype=torch.int32, device=dev)
    off_dev = offsets.to(dev)
    A.check(lib, lib.pgpd_gpd_project(_ptr(pc), P, _ptr(fr), G, _ptr(off_dev), _ptr(idx), chann, _ptr(out), _ptr(valid),
                                      (ws.data_ptr() + 255) & ~255, nbytes, stream))
    return out, valid
