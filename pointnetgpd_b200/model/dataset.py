"""`model.dataset` with the reference's class surface (PointNetGPD/model/dataset.py).

The four datasets the training scripts construct: `PointGraspDataset` (:201-285), `PointGraspMultiClassDataset`
(:288-372), `PointGraspOneViewDataset` (:375-461), `PointGraspOneViewMultiClassDataset` (:464-549).  Same constructor
signatures, same on-disk layout ($PointNetGPD_FOLDER tree, SURVEY.md 7.4), same sample contract:
`(points float64 [3, grasp_points_num], label[, object name])` or `None` for samples the collate function drops.

Written from the reference's behaviour, not its code: one class parameterised by (views, classes).  The gripper-box
crop is `crop_points` below (numpy, runs in DataLoader workers like the reference); the batched GPU version of the
same crop is `pointnetgpd_b200.prep.crop`.

`projection=True` (the GPD baseline scripts, main_1v_gpd.py / main_fullv_gpd.py) yields the reference's 60 x 60 images
instead: `(image float64 [project_chann, 60, 60], label[, object name])` or `None` (dataset.py:88-198,270).  The items
are built on the CPU by `pointnetgpd_b200.projection` (numpy + cKDTree; the workers are forked after the script has
initialised CUDA); `pointnetgpd_b200.prep.project` computes the same images for many grasps of a cloud on the GPU.
"""
import glob
import os
import pickle

import numpy as np
import torch.utils.data

from .. import projection as _projection

__all__ = ["BaseGraspDataset", "PointGraspDataset", "PointGraspMultiClassDataset", "PointGraspOneViewDataset",
           "PointGraspOneViewMultiClassDataset"]


_MMAPS = {}


def _mmap(path):
    """Read-only memory map of a .npy file, cached per process (falls back to np.load for files numpy cannot map)."""
    m = _MMAPS.get(path)
    if m is None:
        try:
            m = np.load(path, mmap_mode="r")
        except ValueError:
            m = np.load(path)
        _MMAPS[path] = m
    return m


def grasp_frame(grasp, transform):
    """(center, rows=(approach, binormal, minor_normal), width) of a 12-float grasp row in the cloud frame."""
    c = np.asarray(grasp[0:3], dtype=np.float64)
    b = np.asarray(grasp[3:6], dtype=np.float64)
    b = b / np.linalg.norm(b)
    width, ang = float(grasp[6]), float(grasp[7])
    ex = np.array([b[1], -b[0], 0.0])
    ex = np.array([1.0, 0.0, 0.0]) if np.linalg.norm(ex) == 0 else ex / np.linalg.norm(ex)
    ez = np.cross(ex, b)
    approach = np.cos(ang) * ex + np.sin(ang) * ez
    approach = approach / np.linalg.norm(approach)
    minor = np.cross(b, approach)
    T = np.asarray(transform, dtype=np.float64)
    R, t = T[:3, :3], T[:3, 3]
    return R @ c + t, np.stack([R @ approach, R @ b, R @ minor]), width


def crop_points(grasp, pc, transform):
    """Indices of the cloud points inside the gripper box and their coordinates in the grasp frame."""
    center, rows, width = grasp_frame(grasp, transform)
    local = (np.asarray(pc) - center) @ rows.T
    half = np.array([width / 4, width / 2, width / 4])
    inside = np.all((local > -half) & (local < half), axis=1)
    idx = np.nonzero(inside)[0]
    return idx, local[idx]


class BaseGraspDataset(torch.utils.data.Dataset):
    min_point_limit = 50

    def __init__(self):
        self.pointnetgpd_dir = os.environ["PointNetGPD_FOLDER"]
        with open(os.path.join(self.pointnetgpd_dir, "PointNetGPD", "data", "google2cloud.pkl"), "rb") as f:
            self.transform = pickle.load(f)
        self.projection = False
        self.in_ind = None

    def collect_pc(self, grasp, pc, transform):
        if self.projection:
            center, rows, width = grasp_frame(grasp, transform)
            self.in_ind, img = _projection.project_grasp(pc, center, rows, width, self.project_chann)
            return None if img is None else img.transpose(2, 1, 0)            # [x, y, c] like project_pc
        self.in_ind, pts = crop_points(grasp, pc, transform)
        return None if len(self.in_ind) < self.min_point_limit else pts


class _GraspDataset(BaseGraspDataset):
    ONE_VIEW = False
    MULTI_CLASS = False

    def _setup(self, grasp_points_num, grasp_amount_per_file, thresh_good, thresh_bad, tag, with_obj, projection,
               project_chann, project_size, obj_points_num=None, pc_file_used_num=None):
        super().__init__()
        if project_chann not in (3, 12) or project_size != 60:
            raise NotImplementedError
        self.obj_points_num, self.pc_file_used_num = obj_points_num, pc_file_used_num
        self.grasp_points_num, self.grasp_amount_per_file = grasp_points_num, grasp_amount_per_file
        self.thresh_good, self.thresh_bad, self.tag, self.with_obj = thresh_good, thresh_bad, tag, with_obj
        self.projection, self.project_chann, self.project_size = projection, project_chann, project_size
        root = self.pointnetgpd_dir
        pattern = "pc_NP3_NP5*.npy" if self.ONE_VIEW else "*.npy"
        self.d_pc = {}
        for f in glob.glob(os.path.join(root, "data", "ycb-tools", "models", "ycb", "*", "rgbd", "clouds", pattern)):
            self.d_pc.setdefault(f.split("/")[-4], []).append(f)
        for v in self.d_pc.values():
            v.sort()
        self.d_grasp = {os.path.basename(f).split(".")[0]: f
                        for f in glob.glob(os.path.join(root, "PointNetGPD", "data", "ycb_grasp", tag, "*.npy"))}
        self.object = sorted(set(self.d_grasp) & set(self.transform))
        self.amount = len(self.object) * grasp_amount_per_file

    def __len__(self):
        return self.amount

    def __getitem__(self, index):
        obj_ind, grasp_ind = np.unravel_index(index, (len(self.object), self.grasp_amount_per_file))
        name = self.object[obj_ind]
        cloud_name, transform = self.transform[name][0], self.transform[name][1]
        files = self.d_pc[cloud_name]
        # memory-mapped reads (SURVEY.md 8f row 3): the reference re-reads and parses the whole 6500 x 12 grasp file and the view
        # clouds for every item; a read-only map touches only the row / pages it uses and is shared by the DataLoader workers
        grasp = np.array(_mmap(self.d_grasp[name])[grasp_ind])
        if self.ONE_VIEW:
            pc = _mmap(files[np.random.randint(len(files))])                        # one random view
        else:
            picks = np.random.choice(len(files), size=self.pc_file_used_num)        # stack views, thin to obj_points_num
            pc = np.vstack([_mmap(files[i]) for i in picks])
            pc = pc[np.random.choice(len(pc), size=self.obj_points_num)]
        pts = self.collect_pc(grasp, pc, transform)
        if pts is None:
            return None
        if self.projection:
            pts = pts.transpose((2, 1, 0))
        else:
            n = len(pts)
            pts = pts[np.random.choice(n, size=self.grasp_points_num, replace=not (n > self.grasp_points_num))].T
        score = grasp[-2] + grasp[-1] * 0.01
        if self.MULTI_CLASS:
            label = 0 if score >= self.thresh_bad else (2 if score <= self.thresh_good else 1)
        else:
            if score >= self.thresh_bad:
                label = 0
            elif score <= self.thresh_good:
                label = 1
            else:
                return None
        return (pts, label, name) if self.with_obj else (pts, label)


class PointGraspDataset(_GraspDataset):
    def __init__(self, obj_points_num, grasp_points_num, pc_file_used_num, grasp_amount_per_file, thresh_good,
                 thresh_bad, tag, with_obj=False, projection=False, project_chann=3, project_size=60):
        self._setup(grasp_points_num, grasp_amount_per_file, thresh_good, thresh_bad, tag, with_obj, projection,
                    project_chann, project_size, obj_points_num, pc_file_used_num)


class PointGraspMultiClassDataset(PointGraspDataset):
    MULTI_CLASS = True


class PointGraspOneViewDataset(_GraspDataset):
    ONE_VIEW = True

    def __init__(self, grasp_points_num, grasp_amount_per_file, thresh_good, thresh_bad, tag, with_obj=False,
                 projection=False, project_chann=3, project_size=60):
        self._setup(grasp_points_num, grasp_amount_per_file, thresh_good, thresh_bad, tag, with_obj, projection,
                    project_chann, project_size)
        self.minimum_point_amount = 150


class PointGraspOneViewMultiClassDataset(PointGraspOneViewDataset):
    MULTI_CLASS = True
