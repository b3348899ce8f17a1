"""CPU test of the torch.autograd glue (pointnetgpd_b200.functional._Fused) and of the nn.Module
surface, with libpgpd swapped for its SIMT-emulator build.  Checks argument order, gradient
routing to the right parameters, buffer updates, and pickle / state_dict compatibility."""
import io
import os
import pickle

import numpy as np
import pytest
import torch

import emu_util as E
from golden_util import load_case, is_zero_grad_param, shipped_state
from oracle import pointnet_torch_port as PT
from pointnetgpd_b200 import _abi as A
from pointnetgpd_b200 import functional as Fn
from pointnetgpd_b200.model.pointnet import PointNetCls, PointNetfeat, STN3d, DualPointNetCls


@pytest.fixture()
def emu(monkeypatch):
    lib = E.emu_lib()
    monkeypatch.setattr(A, "load", lambda: lib)
    return lib


def _load_state(m, np_state):
    m.load_state_dict({k: torch.tensor(v) for k, v in np_state.items()}, strict=True)


def _apply(module, what, x, k=1):
    params, bufs = Fn.gather_tensors(module, what)
    return Fn._Fused.apply(what, bool(module.training), k, 0, x, *params, *bufs)


def test_module_train_step_through_autograd(emu):
    c = load_case("fresh_b8_n96_k2")
    m = PointNetCls(num_points=c["N"], input_chann=3, k=c["k"])
    _load_state(m, c["state"])
    m.train()
    x = torch.tensor(c["x"])
    logp, trans = _apply(m, A.PGPD_CLS, x, k=c["k"])
    loss = torch.nn.functional.nll_loss(logp, torch.tensor(c["y"]))
    loss.backward()
    g = c["g"]
    assert abs(float(loss) - float(g["train_loss_f64"])) < 1e-4
    sd = PT.to_torch_state(c["state"], torch.float32, requires_grad=True)
    _, _, _, ref = PT.train_step(sd, x, torch.tensor(c["y"]))
    for name, p in m.named_parameters():
        assert p.grad is not None and p.grad.shape == p.shape, name
        if is_zero_grad_param(name):
            continue
        r = ref[name]
        assert float((p.grad - r).norm() / r.norm()) < 2e-2, name
    for name, b in m.named_buffers():
        if name.endswith("num_batches_tracked"):
            assert int(b) == 1
        else:
            assert np.allclose(b.numpy(), g["buf_f64/" + name], atol=1e-4), name


def test_misaligned_parameter_views_like_dataparallel_replicas(emu):
    """nn.DataParallel replicas are views into a coalesced broadcast buffer at arbitrary 4-byte offsets
    (torch.nn.parallel.replicate); the C ABI wants 16-byte aligned weights, so the glue must pass aligned copies and the
    gradients must still reach the (misaligned) parameters."""
    c = load_case("fresh_b8_n96_k2")
    m = PointNetCls(num_points=c["N"], input_chann=3, k=c["k"])
    _load_state(m, c["state"])
    ref = PointNetCls(num_points=c["N"], input_chann=3, k=c["k"])
    _load_state(ref, c["state"])
    for name, p in list(m.named_parameters()):
        flat = torch.zeros(p.numel() + 1)
        flat[1:] = p.detach().reshape(-1)
        view = flat[1:].view_as(p)                       # 4 bytes past a 64-byte aligned allocation
        assert view.data_ptr() % 16 != 0
        mod = m
        parts = name.split(".")
        for q in parts[:-1]:
            mod = getattr(mod, q)
        mod._parameters[parts[-1]] = torch.nn.Parameter(view)
    m.train(); ref.train()
    x = torch.tensor(c["x"]); y = torch.tensor(c["y"])
    out = []
    for mm in (m, ref):
        logp, _ = _apply(mm, A.PGPD_CLS, x, k=c["k"])
        torch.nn.functional.nll_loss(logp, y).backward()
        out.append(logp.detach())
    assert torch.equal(out[0], out[1])
    for (n, p), (_, r) in zip(m.named_parameters(), ref.named_parameters()):
        assert p.grad is not None and torch.equal(p.grad, r.grad), n


def test_eval_no_grad_and_eval_backward_raises(emu):
    c = load_case("wild_b6_n80_k3")
    m = PointNetCls(num_points=c["N"], k=c["k"])
    _load_state(m, c["state"])
    m.eval()
    x = torch.tensor(c["x"])
    with torch.no_grad():
        logp, trans = _apply(m, A.PGPD_CLS, x, k=c["k"])
    assert np.abs(logp.numpy() - c["g"]["eval_logp_f64"]).max() < 1e-3
    assert not logp.requires_grad
    logp, _ = _apply(m, A.PGPD_CLS, x, k=c["k"])
    with pytest.raises(NotImplementedError):
        logp.sum().backward()


def test_stn_and_feat_modules_route_gradients(emu):
    c = load_case("wild_b6_n80_k3")
    full = PointNetCls(num_points=c["N"], k=c["k"])
    _load_state(full, c["state"])
    feat = full.feat.train()
    x = torch.tensor(c["x"])
    G, trans = _apply(feat, A.PGPD_FEAT, x)
    assert G.shape == (c["B"], 1024) and trans.shape == (c["B"], 3, 3)
    (G.sum() + trans.sum()).backward()
    assert all(p.grad is not None for p in feat.parameters())
    stn = full.feat.stn
    for p in stn.parameters():
        p.grad = None
    out, trans = _apply(stn, A.PGPD_STN, x)
    trans.square().sum().backward()
    assert all(p.grad is not None and torch.isfinite(p.grad).all() for p in stn.parameters())


def test_product_surface_rejects_what_it_does_not_cover():
    m = PointNetCls(num_points=32, k=2)
    with pytest.raises(RuntimeError, match="CUDA-only"):
        m(torch.zeros(2, 3, 32))
    d = DualPointNetCls(32, 6, 2)                            # constructible; same 111 state_dict keys as the reference class
    from pointnetgpd_b200 import synth
    assert list(d.state_dict().keys()) == synth.state_keys(2, dual=True)
    with pytest.raises(RuntimeError, match="CUDA-only"):
        d(torch.zeros(2, 6, 32))
    from pointnetgpd_b200.model.pointnet import PointNetDenseCls
    with pytest.raises(NotImplementedError):
        PointNetDenseCls()
    from pointnetgpd_b200.model.gpd import GPDClassifier
    g = GPDClassifier(3)                                     # constructible (same sub-modules as the reference); CUDA-only forward
    assert list(g.state_dict().keys()) == ["conv1.weight", "conv1.bias", "conv2.weight", "conv2.bias", "fc1.weight", "fc1.bias",
                                           "fc2.weight", "fc2.bias"]
    with pytest.raises(RuntimeError, match="CUDA-only"):
        g(torch.zeros(2, 3, 60, 60))


def test_state_dict_keys_and_pickle_roundtrip():
    from oracle.weights import state_keys
    m = PointNetCls(num_points=500, k=3)
    assert list(m.state_dict().keys()) == state_keys(3)
    buf = io.BytesIO()
    torch.save(m, buf)                       # whole-module pickle, main_1v.py:178
    buf.seek(0)
    m2 = torch.load(buf, weights_only=False)
    assert isinstance(m2, PointNetCls) and isinstance(m2.feat, PointNetfeat) and isinstance(m2.feat.stn, STN3d)
    for (k1, v1), (k2, v2) in zip(m.state_dict().items(), m2.state_dict().items()):
        assert k1 == k2 and torch.equal(v1, v2)
    # nn.DataParallel wraps it and arbitrary attributes can be set (main_1v.py:154,165)
    m.device_ids = [0]
    dp = torch.nn.DataParallel(m, device_ids=None) if torch.cuda.is_available() else None
    assert m.device_ids == [0]


def test_shipped_checkpoint_unpickles_into_our_classes(golden_dir, tmp_path):
    """The 2018 whole-module pickle references `model.pointnet.{PointNetCls,PointNetfeat,STN3d}` (SURVEY App. B);
    with install_as_model() those resolve to this package's classes, without running __init__.  The file is rebuilt from
    the checkpoint's own object pickle and the tensors of the reduced fixture (oracle/make_golden.py)."""
    import sys
    import types
    import pointnetgpd_b200
    from oracle.make_golden import write_shipped_pickle
    ref = shipped_state()
    fx = np.load(os.path.join(golden_dir, "shipped_3class_pickle.npz"))
    path = str(tmp_path / "pointnetgpd_3class.model")
    write_shipped_pickle(path, fx["head"], fx["storage_keys"], ref)
    saved = {k: sys.modules.get(k) for k in ("model", "model.pointnet", "model.gpd", "torch.nn.backends.thnn")}
    try:
        pointnetgpd_b200.install_as_model(force=True)
        thnn = types.ModuleType("torch.nn.backends.thnn")
        thnn._get_thnn_function_backend = lambda: None
        sys.modules["torch.nn.backends.thnn"] = thnn
        import warnings
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            obj = torch.load(path, map_location="cpu", weights_only=False)
        mod = obj.module if isinstance(obj, torch.nn.DataParallel) else obj
        assert type(mod) is PointNetCls and type(mod.feat.stn) is STN3d
        assert mod.num_points == 500 and mod.fc3.out_features == 3
        for k, v in mod.state_dict().items():
            assert np.array_equal(v.numpy(), ref[k]), k
        params, bufs = Fn.gather_tensors(mod, A.PGPD_CLS)
        assert len(params) == 44 and len(bufs) == 30
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v
