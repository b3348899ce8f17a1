"""ctypes binding of libpgpd.so (C ABI declared in include/pgpd.h).

The library is hand-written sm_100a CUDA built in-tree by `__graft_entry__.build()` /
`pointnetgpd_b200/build.py`.  There is NO fallback: if the shared object is missing or does not
export the ABI, importing the fused path raises -- it never silently routes to PyTorch ops.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libpgpd.so")

PGPD_STN, PGPD_FEAT, PGPD_CLS = 1, 2, 3
F_TRAIN, F_SAVE, F_SIMT = 0x1, 0x2, 0x100
F_BWD_HEAD, F_BWD_STN = 0x10, 0x20
E_ARG, E_WORKSPACE, E_BATCH1, E_CUDA, E_UNSUPPORTED = -1, -2, -3, -4, -5

_fp = C.c_void_p  # device pointers travel as integers


class Lin(C.Structure):
    _fields_ = [("w", _fp), ("b", _fp)]


class Bn(C.Structure):
    _fields_ = [("gamma", _fp), ("beta", _fp), ("running_mean", _fp), ("running_var", _fp),
                ("num_batches_tracked", _fp)]


class Tower(C.Structure):
    _fields_ = [("conv", Lin * 3), ("bn", Bn * 3)]


class Head(C.Structure):
    _fields_ = [("fc", Lin * 3), ("bn", Bn * 2)]


class Model(C.Structure):
    _fields_ = [("stn_tower", Tower), ("stn_head", Head), ("trunk", Tower), ("cls_head", Head)]


class LinGrad(C.Structure):
    _fields_ = [("dw", _fp), ("db", _fp)]


class BnGrad(C.Structure):
    _fields_ = [("dgamma", _fp), ("dbeta", _fp)]


class TowerGrad(C.Structure):
    _fields_ = [("conv", LinGrad * 3), ("bn", BnGrad * 3)]


class HeadGrad(C.Structure):
    _fields_ = [("fc", LinGrad * 3), ("bn", BnGrad * 2)]


class ModelGrad(C.Structure):
    _fields_ = [("stn_tower", TowerGrad), ("stn_head", HeadGrad), ("trunk", TowerGrad), ("cls_head", HeadGrad)]


class Gpd(C.Structure):
    _fields_ = [("conv1", Lin), ("conv2", Lin), ("fc1", Lin), ("fc2", Lin)]


class GpdGrad(C.Structure):
    _fields_ = [("conv1", LinGrad), ("conv2", LinGrad), ("fc1", LinGrad), ("fc2", LinGrad)]


GPD_LAYERS = ("conv1", "conv2", "fc1", "fc2")

# the dual-cloud network (SimpleSTN3d / DualPointNetfeat / DualPointNetCls, pointnet.py:48-120,157-174)
PGPD_DUAL_STN, PGPD_DUAL_FEAT, PGPD_DUAL_CLS = 11, 12, 13


class Dual(C.Structure):
    _fields_ = [("stn1_tower", Tower), ("stn1_head", Head), ("stn2_tower", Tower), ("stn2_head", Head), ("trunk", Tower), ("cls_head", Head)]


class DualGrad(C.Structure):
    _fields_ = [("stn1_tower", TowerGrad), ("stn1_head", HeadGrad), ("stn2_tower", TowerGrad), ("stn2_head", HeadGrad),
                ("trunk", TowerGrad), ("cls_head", HeadGrad)]


EXPORTS = ("pgpd_dual_workspace_bytes", "pgpd_dual_forward", "pgpd_dual_backward", "pgpd_gpd_workspace_bytes", "pgpd_gpd_forward", "pgpd_gpd_backward", "pgpd_version", "pgpd_last_error", "pgpd_has_tensor_core_path", "pgpd_launch_count",
           "pgpd_profile_enable", "pgpd_profile_read", "pgpd_workspace_bytes",
           "pgpd_forward", "pgpd_backward", "pgpd_tower_workspace_bytes", "pgpd_tower_forward",
           "pgpd_tower_backward", "pgpd_crop_box", "pgpd_resample", "pgpd_gpd_project_workspace_bytes", "pgpd_gpd_project")


def bind(lib):
    """Declare argument/return types of every exported symbol on a loaded CDLL."""
    for name in EXPORTS:
        if not hasattr(lib, name):
            raise RuntimeError("libpgpd is missing the symbol %s declared in include/pgpd.h" % name)
    lib.pgpd_version.restype = C.c_int
    lib.pgpd_last_error.restype = C.c_char_p
    lib.pgpd_has_tensor_core_path.restype = C.c_int
    lib.pgpd_launch_count.restype = C.c_ulonglong
    lib.pgpd_profile_enable.restype = C.c_int
    lib.pgpd_profile_enable.argtypes = [C.c_int]
    lib.pgpd_profile_read.restype = C.c_int
    lib.pgpd_profile_read.argtypes = [C.POINTER(C.c_int), C.POINTER(C.c_float)]
    lib.pgpd_workspace_bytes.restype = C.c_size_t
    lib.pgpd_workspace_bytes.argtypes = [C.c_int] * 5
    lib.pgpd_forward.restype = C.c_int
    lib.pgpd_forward.argtypes = [C.c_int, C.POINTER(Model), _fp, C.c_int, C.c_int, C.c_int, C.c_int,
                                 _fp, _fp, _fp, C.c_size_t, _fp]
    lib.pgpd_backward.restype = C.c_int
    lib.pgpd_backward.argtypes = [C.c_int, C.POINTER(Model), C.POINTER(ModelGrad), _fp, C.c_int, C.c_int,
                                  C.c_int, C.c_int, _fp, _fp, _fp, C.c_size_t, _fp]
    lib.pgpd_tower_workspace_bytes.restype = C.c_size_t
    lib.pgpd_tower_workspace_bytes.argtypes = [C.c_int] * 3
    lib.pgpd_tower_forward.restype = C.c_int
    lib.pgpd_tower_forward.argtypes = [C.POINTER(Tower), _fp, _fp, C.c_int, C.c_int, C.c_int, C.c_int, _fp,
                                       _fp, C.c_size_t, _fp]
    lib.pgpd_tower_backward.restype = C.c_int
    lib.pgpd_tower_backward.argtypes = [C.POINTER(Tower), C.POINTER(TowerGrad), _fp, _fp, C.c_int, C.c_int,
                                        C.c_int, C.c_int, _fp, _fp, _fp, C.c_size_t, _fp]
    lib.pgpd_gpd_workspace_bytes.restype = C.c_size_t
    lib.pgpd_gpd_workspace_bytes.argtypes = [C.c_int] * 3
    lib.pgpd_gpd_forward.restype = C.c_int
    lib.pgpd_gpd_forward.argtypes = [C.POINTER(Gpd), _fp, C.c_int, C.c_int, C.c_int, _fp, _fp, C.c_size_t, _fp]
    lib.pgpd_gpd_backward.restype = C.c_int
    lib.pgpd_gpd_backward.argtypes = [C.POINTER(Gpd), C.POINTER(GpdGrad), _fp, C.c_int, C.c_int, C.c_int, _fp, _fp, C.c_size_t, _fp]
    lib.pgpd_dual_workspace_bytes.restype = C.c_size_t
    lib.pgpd_dual_workspace_bytes.argtypes = [C.c_int] * 5
    lib.pgpd_dual_forward.restype = C.c_int
    lib.pgpd_dual_forward.argtypes = [C.c_int, C.POINTER(Dual), _fp, C.c_int, C.c_int, C.c_int, C.c_int, _fp, _fp, _fp, C.c_size_t, _fp]
    lib.pgpd_dual_backward.restype = C.c_int
    lib.pgpd_dual_backward.argtypes = [C.c_int, C.POINTER(Dual), C.POINTER(DualGrad), _fp, C.c_int, C.c_int, C.c_int,
                                       C.c_int, _fp, _fp, _fp, C.c_size_t, _fp]
    lib.pgpd_crop_box.restype = C.c_int
    lib.pgpd_crop_box.argtypes = [_fp, C.c_int, _fp, C.c_int, _fp, _fp, _fp, _fp, _fp]
    lib.pgpd_resample.restype = C.c_int
    lib.pgpd_resample.argtypes = [_fp, _fp, C.c_int, C.c_int, C.c_int, C.c_ulonglong, _fp, _fp, _fp]
    lib.pgpd_gpd_project_workspace_bytes.restype = C.c_size_t
    lib.pgpd_gpd_project_workspace_bytes.argtypes = [C.c_int] * 4
    lib.pgpd_gpd_project.restype = C.c_int
    lib.pgpd_gpd_project.argtypes = [_fp, C.c_int, _fp, C.c_int, _fp, _fp, C.c_int, _fp, _fp, _fp, C.c_size_t, _fp]
    return lib


_lib = None


def load():
    """Load (once) and return the product library.  Raises if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                "pointnetgpd_b200: %s not found -- build it with `python -m pointnetgpd_b200.build` "
                "(nvcc, sm_100a).  There is no non-CUDA fallback for the fused PointNet path." % LIB_PATH)
        _lib = bind(C.CDLL(LIB_PATH))
    return _lib


class PgpdError(RuntimeError):
    pass


def check(lib, rc):
    """Map a negative return code to the exception the reference would raise."""
    if rc == 0:
        return
    msg = lib.pgpd_last_error().decode()
    if rc == E_BATCH1:
        # what torch.nn.functional.batch_norm raises for a train-mode batch of 1 (SURVEY.md 7.2 E)
        raise ValueError(msg)
    if rc == E_ARG:
        raise ValueError("pgpd: " + msg)
    raise PgpdError("pgpd error %d: %s" % (rc, msg))


# ---- state-dict key -> struct field mapping (key names of the reference PointNetCls, SURVEY.md 8b) ----
def _tower_keys(prefix):
    return [(prefix + "conv%d" % (i + 1), prefix + "bn%d" % (i + 1)) for i in range(3)]


TOWER_STN, TOWER_TRUNK = "feat.stn.", "feat."
HEAD_STN = ("feat.stn.", ("bn4", "bn5"))
HEAD_CLS = ("", ("bn1", "bn2"))


def fill_tower(t, prefix, ptr):
    for i, (conv, bn) in enumerate(_tower_keys(prefix)):
        t.conv[i].w, t.conv[i].b = ptr(conv + ".weight"), ptr(conv + ".bias")
        _fill_bn(t.bn[i], bn, ptr)


def _fill_bn(b, name, ptr):
    b.gamma, b.beta = ptr(name + ".weight"), ptr(name + ".bias")
    b.running_mean, b.running_var = ptr(name + ".running_mean"), ptr(name + ".running_var")
    b.num_batches_tracked = ptr(name + ".num_batches_tracked")


def fill_head(h, spec, ptr):
    prefix, bns = spec
    for i in range(3):
        h.fc[i].w, h.fc[i].b = ptr(prefix + "fc%d.weight" % (i + 1)), ptr(prefix + "fc%d.bias" % (i + 1))
    for i, bn in enumerate(bns):
        _fill_bn(h.bn[i], prefix + bn, ptr)


def build_model(ptr, what=PGPD_CLS):
    """ptr(key) -> device address (int) of the tensor stored under state-dict key `key`."""
    m = Model()
    fill_tower(m.stn_tower, TOWER_STN, ptr)
    fill_head(m.stn_head, HEAD_STN, ptr)
    if what >= PGPD_FEAT:
        fill_tower(m.trunk, TOWER_TRUNK, ptr)
    if what == PGPD_CLS:
        fill_head(m.cls_head, HEAD_CLS, ptr)
    return m


def fill_tower_grad(t, prefix, ptr):
    for i, (conv, bn) in enumerate(_tower_keys(prefix)):
        t.conv[i].dw, t.conv[i].db = ptr(conv + ".weight"), ptr(conv + ".bias")
        t.bn[i].dgamma, t.bn[i].dbeta = ptr(bn + ".weight"), ptr(bn + ".bias")


def fill_head_grad(h, spec, ptr):
    prefix, bns = spec
    for i in range(3):
        h.fc[i].dw, h.fc[i].db = ptr(prefix + "fc%d.weight" % (i + 1)), ptr(prefix + "fc%d.bias" % (i + 1))
    for i, bn in enumerate(bns):
        h.bn[i].dgamma, h.bn[i].dbeta = ptr(prefix + bn + ".weight"), ptr(prefix + bn + ".bias")


def build_grads(ptr, what=PGPD_CLS):
    g = ModelGrad()
    fill_tower_grad(g.stn_tower, TOWER_STN, ptr)
    fill_head_grad(g.stn_head, HEAD_STN, ptr)
    if what >= PGPD_FEAT:
        fill_tower_grad(g.trunk, TOWER_TRUNK, ptr)
    if what == PGPD_CLS:
        fill_head_grad(g.cls_head, HEAD_CLS, ptr)
    return g


def param_keys(what=PGPD_CLS, k=None):
    """Parameter keys (the ones that receive gradients) a module owns, in a fixed order."""
    keys = []
    def tower(prefix):
        for conv, bn in _tower_keys(prefix):
            keys.extend([conv + ".weight", conv + ".bias", bn + ".weight", bn + ".bias"])
    def head(spec):
        prefix, bns = spec
        for i in range(3):
            keys.extend([prefix + "fc%d.weight" % (i + 1), prefix + "fc%d.bias" % (i + 1)])
        for bn in bns:
            keys.extend([prefix + bn + ".weight", prefix + bn + ".bias"])
    tower(TOWER_STN)
    head(HEAD_STN)
    if what >= PGPD_FEAT:
        tower(TOWER_TRUNK)
    if what == PGPD_CLS:
        head(HEAD_CLS)
    return keys


def buffer_keys(what=PGPD_CLS):
    keys = []
    def bn(name):
        keys.extend([name + ".running_mean", name + ".running_var", name + ".num_batches_tracked"])
    for _c, b in _tower_keys(TOWER_STN):
        bn(b)
    for b in HEAD_STN[1]:
        bn(HEAD_STN[0] + b)
    if what >= PGPD_FEAT:
        for _c, b in _tower_keys(TOWER_TRUNK):
            bn(b)
    if what == PGPD_CLS:
        for b in HEAD_CLS[1]:
            bn(HEAD_CLS[0] + b)
    return keys


# ---- the dual-cloud network: module-relative key prefixes per sub-struct ------------------------------------------------------------
#   PGPD_DUAL_CLS keys are DualPointNetCls-relative ("feat.stn1.conv1.weight", ..., "fc3.bias"); stand-alone DualPointNetfeat /
#   SimpleSTN3d modules strip "feat." / use no prefix at all (see functional.run_dual).
_DUAL_STN_HEAD_BNS = ("bn4", "bn5")


def _dual_parts(what):
    """[(struct field, kind, key prefix, head BatchNorm names)] of the sub-structs a module owns, in ABI order."""
    if what == PGPD_DUAL_STN:
        return [("stn1_tower", "tower", "", None), ("stn1_head", "head", "", _DUAL_STN_HEAD_BNS)]
    pre = "feat." if what == PGPD_DUAL_CLS else ""
    parts = []
    for i in (1, 2):
        parts += [("stn%d_tower" % i, "tower", pre + "stn%d." % i, None), ("stn%d_head" % i, "head", pre + "stn%d." % i, _DUAL_STN_HEAD_BNS)]
    parts.append(("trunk", "tower", pre, None))
    if what == PGPD_DUAL_CLS:
        parts.append(("cls_head", "head", "", ("bn1", "bn2")))
    return parts


def build_dual(ptr, what, grad=False):
    """ptr(key) -> device address of the tensor (grad: of its gradient) stored under the module-relative state-dict key."""
    m = DualGrad() if grad else Dual()
    for field, kind, prefix, bns in _dual_parts(what):
        sub = getattr(m, field)
        if kind == "tower":
            (fill_tower_grad if grad else fill_tower)(sub, prefix, ptr)
        else:
            (fill_head_grad if grad else fill_head)(sub, (prefix, bns), ptr)
    return m


def dual_param_keys(what):
    keys = []
    for _f, kind, prefix, bns in _dual_parts(what):
        if kind == "tower":
            for conv, bn in _tower_keys(prefix):
                keys.extend([conv + ".weight", conv + ".bias", bn + ".weight", bn + ".bias"])
        else:
            for i in range(3):
                keys.extend([prefix + "fc%d.weight" % (i + 1), prefix + "fc%d.bias" % (i + 1)])
            for bn in bns:
                keys.extend([prefix + bn + ".weight", prefix + bn + ".bias"])
    return keys


def dual_buffer_keys(what):
    keys = []
    for _f, kind, prefix, bns in _dual_parts(what):
        names = [b for _c, b in _tower_keys(prefix)] if kind == "tower" else [prefix + b for b in bns]
        for name in names:
            keys.extend([name + ".running_mean", name + ".running_var", name + ".num_batches_tracked"])
    return keys
