#!/usr/bin/env python
"""Generate tests/golden/*.npz by running the UNMODIFIED reference module.

TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).

Run where a checkout of the reference project is available:
    python oracle/make_golden.py /path/to/reference-checkout
(the directory that holds PointNetGPD/ and data/).  It imports PointNetGPD/model/pointnet.py (PointNetCls, :177-194),
loads deterministic weights from oracle.weights, runs forward / nll_loss /
backward exactly as main_1v.py:72-75 does, and stores inputs-by-recipe plus
outputs.  Nothing is copied from the reference: the fixtures hold numbers only.

Also reduces the shipped checkpoint (data/pointnetgpd_3class.model, a pickled
DataParallel(PointNetCls(num_points=500, k=3)), SURVEY.md Appendix B) to a fixture
under 1 MB (run_shipped) and records the reference's outputs on it, so that the
real-statistics known-answer tests run without the reference.
"""
import os
import sys
import types

import numpy as np
import torch
import torch.nn.functional as F

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
from oracle import weights as W  # noqa: E402

REF_ROOT = None        # the reference checkout, set by main()
REF = None             # REF_ROOT/PointNetGPD
GOLD = os.path.join(ROOT, "tests", "golden")

# (name, B, N, k, weight style, cloud kind, seed)
CASES = [
    ("fresh_b8_n96_k2", 8, 96, 2, "default", "box", 11),
    ("wild_b6_n80_k3", 6, 80, 3, "wild", "dup", 12),
    ("wild_b5_n200_k2_randn", 5, 200, 2, "wild", "randn", 13),
    ("fresh_b32_n750_k2", 32, 750, 2, "default", "box", 14),   # BASELINE config 1 shape
]

SUBSAMPLE = 97  # entries kept per large gradient tensor


def _import_reference():
    sys.path.insert(0, REF)
    # the shipped 2018 pickle needs this long-gone module (SURVEY.md Appendix B)
    thnn = types.ModuleType("torch.nn.backends.thnn")
    thnn._get_thnn_function_backend = lambda: None
    sys.modules["torch.nn.backends.thnn"] = thnn
    from model.pointnet import PointNetCls  # noqa
    return PointNetCls


def sub_idx(n):
    """Deterministic subsample positions for a flat tensor of n entries."""
    if n <= SUBSAMPLE:
        return np.arange(n)
    return (np.arange(SUBSAMPLE, dtype=np.int64) * 2654435761 % n).astype(np.int64)


def load_state(model, np_state):
    sd = {}
    for k, v in np_state.items():
        sd[k] = torch.tensor(v)
    model.load_state_dict(sd, strict=True)


def run_case(PointNetCls, name, B, N, k, style, kind, seed):
    st = W.make_state(seed, k=k, style=style)
    x = W.make_clouds(seed + 1000, B, N, kind)
    y = W.make_labels(seed + 2000, B, k)
    out = {"meta": np.array([B, N, k, seed], dtype=np.int64),
           "style": np.array(style), "kind": np.array(kind)}

    for dtype, tag in ((torch.float32, "f32"), (torch.float64, "f64")):
        m = PointNetCls(num_points=N, input_chann=3, k=k)
        load_state(m, st)
        m = m.to(dtype)
        xt = torch.tensor(x).to(dtype)
        yt = torch.tensor(y)
        # ---- eval forward with the initial running stats (main_test.py:59-69 path)
        m.eval()
        with torch.no_grad():
            logp_e, trans_e = m(xt)
        out[f"eval_logp_{tag}"] = logp_e.numpy()
        out[f"eval_trans_{tag}"] = trans_e.numpy()
        # ---- one training step (main_1v.py:72-75)
        m.train()
        m.zero_grad()
        logp, trans = m(xt)
        loss = F.nll_loss(logp, yt)
        loss.backward()
        out[f"train_logp_{tag}"] = logp.detach().numpy()
        out[f"train_trans_{tag}"] = trans.detach().numpy()
        out[f"train_loss_{tag}"] = loss.detach().numpy()
        for pname, p in m.named_parameters():
            g = p.grad.detach().numpy().reshape(-1)
            out[f"gnorm_{tag}/{pname}"] = np.array(np.linalg.norm(g.astype(np.float64)))
            out[f"gsub_{tag}/{pname}"] = g[sub_idx(g.size)]
        for bname, b in m.named_buffers():
            if bname.endswith("num_batches_tracked"):
                out[f"buf_{tag}/{bname}"] = b.numpy()
            else:
                out[f"buf_{tag}/{bname}"] = b.detach().numpy()
        # ---- a second output-gradient pattern that also drives d(trans) (autograd generality)
        m.zero_grad()
        load_state(m, st)
        m = m.to(dtype)
        m.train()
        logp, trans = m(xt)
        wl = torch.tensor(W.normal(seed + 3000, (B, k))).to(dtype)
        wt = torch.tensor(W.normal(seed + 4000, (B, 3, 3))).to(dtype)
        ((logp * wl).sum() + (trans * wt).sum()).backward()
        for pname, p in m.named_parameters():
            g = p.grad.detach().numpy().reshape(-1)
            out[f"g2norm_{tag}/{pname}"] = np.array(np.linalg.norm(g.astype(np.float64)))
            out[f"g2sub_{tag}/{pname}"] = g[sub_idx(g.size)]
    np.savez_compressed(os.path.join(GOLD, name + ".npz"), **out)
    print("wrote", name, "loss f32 %.7f f64 %.12f" % (out["train_loss_f32"], out["train_loss_f64"]))


# The six largest matrices of the shipped checkpoint (1.57 M of its 1.61 M values) do not fit a 1 MB fixture.  The fixture
# keeps every other tensor exactly (BatchNorm statistics with negative gammas and extreme running variances, biases, the
# first two convolutions, the last FC layers) and replaces these by seeded draws with each output row's mean and std.
SHIPPED_BIG = ("feat.stn.conv3.weight", "feat.stn.fc1.weight", "feat.stn.fc2.weight", "feat.conv3.weight", "fc1.weight",
               "fc2.weight")


def load_shipped_state(path):
    """The 74-entry state dict of the reduced shipped checkpoint stored at `path` (tests/golden/shipped_3class_state.npz)."""
    z = np.load(path)
    sd = {k: z[k] for k in z.files if "/" not in k}
    for i, k in enumerate(SHIPPED_BIG):
        mean, std = z["rowmean/" + k], z["rowstd/" + k]
        shape = tuple(int(n) for n in z["shape/" + k])
        rows = mean[:, None] + std[:, None] * W.normal(9000 + i, (shape[0], int(np.prod(shape[1:]))))
        sd[k] = rows.reshape(shape).astype(np.float32)
    return sd


def write_shipped_pickle(path, head, storage_keys, sd):
    """Reassemble the legacy torch.save file of the shipped checkpoint from its object pickle (`head`: everything up to the
    table of storages) and the tensors of `sd`, each storage written as torch's legacy format does: int64 numel, raw data."""
    with open(path, "wb") as f:
        f.write(head.tobytes())
        for key in storage_keys:
            v = np.ascontiguousarray(sd[str(key)])
            f.write(np.int64(v.size).tobytes())
            f.write(v.tobytes())


def _shipped_pickle_head(path, sd):
    """The checkpoint's legacy-format header and object pickle, with the class source texts and file paths torch.save
    embedded in it blanked (torch.load only compares them to warn about changed sources), and the state key of every
    storage in file order."""
    import pickle
    import pickletools
    with open(path, "rb") as f:
        for _ in range(3):                      # magic number, protocol version, sys_info
            pickle.load(f)
        obj_start = f.tell()
        blank = set()

        class Probe(pickle.Unpickler):
            def find_class(self, mod, name):
                return super().find_class(mod, name) if mod == "collections" else type(name, (), {"__init__": lambda s, *a, **k: None, "__setstate__": lambda s, st: None})

            def persistent_load(self, pid):
                if pid[0] == "module":
                    blank.update(x for x in pid[2:] if x)
                    return pid[1]
                return None
        Probe(f).load()
        obj_end = f.tell()
        keys = pickle.load(f)
        data_start = f.tell()
        f.seek(0)
        raw = f.read()
    obj = bytearray(raw[obj_start:obj_end])
    for op, arg, pos in reversed(list(pickletools.genops(bytes(obj)))):
        if op.name == "BINUNICODE" and arg in blank:
            obj[pos:pos + 5 + len(arg.encode("utf-8"))] = b"X\x00\x00\x00\x00"
    head = raw[:obj_start] + bytes(obj) + raw[obj_end:data_start]
    # storage -> state key, by content (tensors with equal contents are interchangeable)
    order, off = [], data_start
    for _key in keys:
        n = int(np.frombuffer(raw[off:off + 8], np.int64)[0])
        off += 8
        for name, v in sd.items():
            if v.size == n and raw[off:off + v.nbytes] == np.ascontiguousarray(v).tobytes():
                order.append(name)
                off += v.nbytes
                break
        else:
            raise RuntimeError("storage %s matches no state tensor" % _key)
    assert off == len(raw)
    return np.frombuffer(head, np.uint8), np.array(order)


def run_shipped(PointNetCls):
    path = os.path.join(REF_ROOT, "data", "pointnetgpd_3class.model")
    model = torch.load(path, map_location="cpu", weights_only=False)   # main_test.py:42
    if isinstance(model, torch.nn.DataParallel):                         # main_test.py:55-56
        model = model.module
    full = {k: v.numpy() for k, v in model.state_dict().items()}
    fx = {k: v for k, v in full.items() if k not in SHIPPED_BIG}
    for k in SHIPPED_BIG:
        rows = full[k].astype(np.float64).reshape(full[k].shape[0], -1)
        fx["rowmean/" + k], fx["rowstd/" + k] = rows.mean(1).astype(np.float32), rows.std(1).astype(np.float32)
        fx["shape/" + k] = np.array(full[k].shape, np.int64)
    gold_state = os.path.join(GOLD, "shipped_3class_state.npz")
    np.savez_compressed(gold_state, **fx)
    sd_np = load_shipped_state(gold_state)
    head, order = _shipped_pickle_head(path, full)
    np.savez_compressed(os.path.join(GOLD, "shipped_3class_pickle.npz"), head=head, storage_keys=order)
    sd = {k: torch.tensor(v) for k, v in sd_np.items()}
    out = {}
    for dtype, tag in ((torch.float32, "f32"), (torch.float64, "f64")):
        m = PointNetCls(num_points=500, input_chann=3, k=3)               # modern torch needs attributes 0.4-era pickles lack
        m.load_state_dict(sd)
        m = m.to(dtype).eval()
        for kind, seed in (("box", 123), ("dup", 124)):
            x = W.make_clouds(seed, 8, 500, kind)
            with torch.no_grad():
                logp, trans = m(torch.tensor(x).to(dtype))
            out[f"{kind}_logp_{tag}"] = logp.numpy()
            out[f"{kind}_trans_{tag}"] = trans.numpy()
        # deploy shape: B=1 (kinect2grasp.py:479 / main_test.py:59-69)
        x1 = W.make_clouds(125, 1, 500, "box")
        with torch.no_grad():
            logp, trans = m(torch.tensor(x1).to(dtype))
        out[f"b1_logp_{tag}"] = logp.numpy()
    np.savez_compressed(os.path.join(GOLD, "shipped_3class_outputs.npz"), **out)
    print("wrote shipped checkpoint fixtures; box logp[0] =", out["box_logp_f32"][0])


def run_collect_pc():
    """Golden vectors for the gripper-box crop: executes the reference's own BaseGraspDataset.collect_pc
    (PointNetGPD/model/dataset.py:15-76).  dataset.py cannot be imported here (it needs open3d), so the method's
    source is pulled out of the file with `ast` and executed as is against a stub `self` -- nothing is copied."""
    import ast
    path = os.path.join(REF, "model", "dataset.py")
    src = open(path).read()
    fn = None
    for node in ast.walk(ast.parse(src)):
        if isinstance(node, ast.FunctionDef) and node.name == "collect_pc":
            fn = ast.get_source_segment(src, node)
            break
    ns = {"np": np}
    import textwrap
    exec(textwrap.dedent(fn), ns)
    stub = types.SimpleNamespace(min_point_limit=1, projection=False, in_ind=None)
    P, G, seed = 4000, 9, 77
    pc = W.uniform(seed, (P, 3), -0.12, 0.12).astype(np.float32)
    centers = W.uniform(seed + 1, (G, 3), -0.05, 0.05)
    axes = W.normal(seed + 2, (G, 3))
    axes[0] = [0, 0, 1.0]
    width = W.uniform(seed + 3, (G,), 0.05, 0.085)
    angle = W.uniform(seed + 4, (G,), -1.5, 1.5)
    grasps = np.concatenate([centers, axes, width[:, None], angle[:, None], np.zeros((G, 4))], axis=1)
    th = 0.3
    T = np.eye(4)
    T[:3, :3] = [[np.cos(th), -np.sin(th), 0], [np.sin(th), np.cos(th), 0], [0, 0, 1]]
    T[:3, 3] = [0.01, -0.02, 0.005]
    out = {"pc": pc, "grasps": grasps, "transform": T}
    for g in range(G):
        res = ns["collect_pc"](stub, grasps[g], pc, T)
        out[f"in_ind_{g}"] = np.asarray(stub.in_ind, dtype=np.int64)
        out[f"pc_t_{g}"] = np.zeros((0, 3)) if res is None else np.asarray(res, dtype=np.float64)
    np.savez_compressed(os.path.join(GOLD, "collect_pc.npz"), **out)
    print("wrote collect_pc golden:", [len(out[f"in_ind_{g}"]) for g in range(G)])


def run_dual(only=False):
    """DualPointNetCls(input_chann=6) (model/pointnet.py:157-174) on two seeded clouds per grasp: eval forward, and a training
    forward + backward of sum(logp * wl) + sum(trans * wt)."""
    from model.pointnet import DualPointNetCls
    B, N, k, seed = 6, 72, 2, 41
    st = W.make_state(seed, k=k, style="wild", dual=True)
    x = np.concatenate([W.make_clouds(seed + 1000, B, N, "box"), W.make_clouds(seed + 1000 + 77, B, N, "box")], axis=1)
    out = {"meta": np.array([B, N, k, seed], dtype=np.int64)}
    for dtype, tag in ((torch.float32, "f32"), (torch.float64, "f64")):
        m = DualPointNetCls(num_points=N, input_chann=6, k=k)
        load_state(m, st)
        m = m.to(dtype)
        xt = torch.tensor(x).to(dtype)
        m.eval()
        with torch.no_grad():
            logp_e, trans_e = m(xt)
        out[f"eval_logp_{tag}"] = logp_e.numpy()
        out[f"eval_trans_{tag}"] = trans_e.numpy()
        m.train()
        m.zero_grad()
        logp, trans = m(xt)
        wl = torch.tensor(W.normal(seed + 3000, (B, k))).to(dtype)
        wt = torch.tensor(W.normal(seed + 4000, (B, 3, 3))).to(dtype)
        ((logp * wl).sum() + (trans * wt).sum()).backward()
        out[f"train_logp_{tag}"] = logp.detach().numpy()
        out[f"train_trans_{tag}"] = trans.detach().numpy()
        for pname, p in m.named_parameters():
            g = p.grad.detach().numpy().reshape(-1)
            out[f"gnorm_{tag}/{pname}"] = np.array(np.linalg.norm(g.astype(np.float64)))
            out[f"gsub_{tag}/{pname}"] = g[sub_idx(g.size)]
        for bname, b in m.named_buffers():
            out[f"buf_{tag}/{bname}"] = b.detach().numpy()
    np.savez_compressed(os.path.join(GOLD, "dual_b6_n72_k2.npz"), **out)
    print("wrote dual_b6_n72_k2; eval logp[0] =", out["eval_logp_f32"][0])


def run_dual_pin():
    """The reference DualPointNetCls on the inputs of tests/test_dual.py::test_dual_port_matches_reference: its state-dict
    keys, eval and train-mode outputs in fp32, and the BatchNorm buffers after the train-mode forward."""
    from model.pointnet import DualPointNetCls
    st = W.make_state(3, k=3, style="wild", dual=True)
    m = DualPointNetCls(40, 6, 3)
    out = {"state_keys": np.array(list(m.state_dict().keys()))}
    load_state(m, st)
    x = torch.tensor(np.concatenate([W.make_clouds(1, 5, 40, "box"), W.make_clouds(1 + 77, 5, 40, "box")], axis=1))
    for training, tag in ((False, "eval"), (True, "train")):
        m.train(training)
        logp, trans = m(x)
        out[f"{tag}_logp"], out[f"{tag}_trans"] = logp.detach().numpy(), trans.detach().numpy()
    for name, b in m.named_buffers():
        out["buf/" + name] = b.numpy()
    np.savez_compressed(os.path.join(GOLD, "dual_pin_b5_n40_k3.npz"), **out)
    print("wrote dual_pin_b5_n40_k3")


def run_gpd_pin():
    """The reference GPDClassifier (PointNetGPD/model/gpd.py) in eval mode on the inputs of
    tests/test_gpd.py::test_gpd_port_matches_reference, and its state-dict keys."""
    import importlib.util
    from oracle import gpd_torch_port as G
    spec = importlib.util.spec_from_file_location("ref_gpd", os.path.join(REF, "model", "gpd.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    out = {"state_keys": np.array(list(mod.GPDClassifier(3).state_dict().keys()))}
    for Cc in (3, 12):
        m = mod.GPDClassifier(Cc)
        m.load_state_dict(G.make_gpd_state(5, Cc))
        m.eval()
        x = torch.tensor(W.normal(6, (3, Cc, 60, 60)).astype(np.float32))
        with torch.no_grad():
            out[f"logp_c{Cc}"] = m(x).numpy()
    np.savez_compressed(os.path.join(GOLD, "gpd_pin.npz"), **out)
    print("wrote gpd_pin")


def main():
    global REF_ROOT, REF
    if len(sys.argv) < 2 or not os.path.isdir(os.path.join(sys.argv[1], "PointNetGPD")):
        raise SystemExit("usage: python oracle/make_golden.py REFERENCE_CHECKOUT [--dual-only]")
    REF_ROOT = os.path.abspath(sys.argv[1])
    REF = os.path.join(REF_ROOT, "PointNetGPD")
    os.makedirs(GOLD, exist_ok=True)
    torch.set_num_threads(8)
    PointNetCls = _import_reference()
    run_dual()
    if "--dual-only" in sys.argv:
        return
    for case in CASES:
        run_case(PointNetCls, *case)
    run_shipped(PointNetCls)
    run_collect_pc()
    run_dual_pin()
    run_gpd_pin()


if __name__ == "__main__":
    main()
