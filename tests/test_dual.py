"""The dual-cloud network -- SimpleSTN3d, DualPointNetfeat, DualPointNetCls (PointNetGPD/model/pointnet.py:48-120,157-174; SURVEY.md
8f row 4): the CUDA implementation (csrc/dual.cuh) against the oracle's torch port -- on the CPU through the SIMT emulator build of
libpgpd (C ABI, numpy buffers), on the GPU through the nn.Module classes.  The port is pinned to the unmodified reference classes
through the reference-generated fixtures tests/golden/dual_pin_b5_n40_k3.npz and dual_b6_n72_k2.npz."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from emu_util import emu_lib, Guarded
from oracle import dual_torch_port as D
from oracle import pointnet_torch_port as P
from pointnetgpd_b200 import _abi as A
from pointnetgpd_b200 import synth as W

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "dual_b6_n72_k2.npz")
PIN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "dual_pin_b5_n40_k3.npz")
STRIP = {A.PGPD_DUAL_CLS: "", A.PGPD_DUAL_FEAT: "feat.", A.PGPD_DUAL_STN: "feat.stn1."}


def dual_clouds(seed, B, N, kind="box"):
    """[B,6,N]: two independent 3-channel clouds per grasp."""
    return np.concatenate([W.make_clouds(seed, B, N, kind), W.make_clouds(seed + 77, B, N, kind)], axis=1)


def sub_state(st, what):
    """Module-relative state of the sub-module `what` from a DualPointNetCls state dict."""
    strip = STRIP[what]
    keys = set(A.dual_param_keys(what)) | set(A.dual_buffer_keys(what))
    return {k[len(strip):]: v for k, v in st.items() if k.startswith(strip) and k[len(strip):] in keys}


def port_forward(sd, x, what, training):
    if what == A.PGPD_DUAL_CLS:
        return D.dual_cls_forward(sd, x, training)
    if what == A.PGPD_DUAL_FEAT:
        return D.dual_feat_forward(sd, x, "", training)
    return None, D.simple_stn3d_forward(sd, x, "", training)


def port_run(st, x, what, training, wo=None, wt=None, dtype=torch.float64):
    """Reference-equivalent outputs (and, with weights wo / wt of a scalar objective sum(out*wo) + sum(trans*wt), gradients)."""
    sd = P.to_torch_state(st, dtype=dtype, requires_grad=wt is not None)
    out, trans = port_forward(sd, torch.tensor(x).to(dtype), what, training)
    grads = None
    if wt is not None:
        obj = (trans * torch.tensor(wt).to(dtype)).sum()
        if out is not None:
            obj = obj + (out * torch.tensor(wo).to(dtype)).sum()
        obj.backward()
        grads = {k: v.grad.numpy() for k, v in sd.items() if v.requires_grad}
    return (None if out is None else out.detach().numpy()), trans.detach().numpy(), grads, sd


def emu_run(st, x, what, training, k, wo=None, wt=None):
    lib = emu_lib()
    st = {kk: np.ascontiguousarray(v).reshape(max(1, v.size)) if v.ndim == 0 else np.ascontiguousarray(v) for kk, v in st.items()}
    B, _, N = x.shape
    x = np.ascontiguousarray(x, np.float32)
    backward = wt is not None
    flags = (A.F_TRAIN if training else 0) | (A.F_SAVE if backward else 0)
    m = A.build_dual(lambda key: st[key].ctypes.data, what)
    nbytes = lib.pgpd_dual_workspace_bytes(what, B, N, k, flags)
    ws = Guarded(nbytes)
    width = {A.PGPD_DUAL_CLS: k, A.PGPD_DUAL_FEAT: 1024, A.PGPD_DUAL_STN: 1}[what]
    out = np.full((B, width), np.nan, np.float32)
    trans = np.full((B, 3, 3), np.nan, np.float32)
    A.check(lib, lib.pgpd_dual_forward(what, C.byref(m), x.ctypes.data, B, N, k, flags, out.ctypes.data, trans.ctypes.data, ws.addr, nbytes, None))
    ws.check()
    grads = None
    if backward:
        grads = {key: np.full(st[key].shape, np.nan, np.float32) for key in A.dual_param_keys(what)}
        g = A.build_dual(lambda key: grads[key].ctypes.data, what, grad=True)
        wo = None if wo is None else np.ascontiguousarray(wo, np.float32)
        wt = np.ascontiguousarray(wt, np.float32)
        A.check(lib, lib.pgpd_dual_backward(what, C.byref(m), C.byref(g), x.ctypes.data, B, N, k, flags,
                                            None if what == A.PGPD_DUAL_STN else wo.ctypes.data, wt.ctypes.data, ws.addr, nbytes, None))
        ws.check()
    return out, trans, grads, st


def rel(a, b):
    return float(np.linalg.norm(a.astype(np.float64) - b) / max(np.linalg.norm(b), 1e-30))


def test_dual_port_matches_reference():
    """Against what the unmodified reference DualPointNetCls computed on the same inputs (oracle/make_golden.py)."""
    gd = np.load(PIN)
    st = W.make_state(3, k=3, style="wild", dual=True)
    assert list(gd["state_keys"]) == W.state_keys(3, dual=True)
    x = torch.tensor(dual_clouds(1, 5, 40))
    for training, tag in ((False, "eval"), (True, "train")):
        sd = P.to_torch_state(st)
        b = D.dual_cls_forward(sd, x, training)
        assert torch.equal(torch.tensor(gd[f"{tag}_logp"]), b[0]) and torch.equal(torch.tensor(gd[f"{tag}_trans"]), b[1])
        if training:
            assert all(torch.equal(torch.tensor(gd["buf/" + k] if "buf/" + k in gd else st[k]), sd[k]) for k in sd)


def test_dual_port_matches_golden():
    """The fixture was written by oracle/make_golden.py from the unmodified reference DualPointNetCls."""
    gd = np.load(GOLD)
    B, N, k, seed = [int(v) for v in gd["meta"]]
    st = W.make_state(seed, k=k, style="wild", dual=True)
    x = dual_clouds(seed + 1000, B, N)
    out, trans, _, _ = port_run(st, x, A.PGPD_DUAL_CLS, False, dtype=torch.float32)
    assert np.array_equal(out, gd["eval_logp_f32"]) and np.array_equal(trans, gd["eval_trans_f32"])
    wo, wt = W.normal(seed + 3000, (B, k)), W.normal(seed + 4000, (B, 3, 3))
    out, trans, grads, sd = port_run(st, x, A.PGPD_DUAL_CLS, True, wo, wt, dtype=torch.float64)
    assert np.abs(out - gd["train_logp_f64"]).max() < 1e-12
    for key, g in grads.items():
        assert abs(np.linalg.norm(g) - gd["gnorm_f64/" + key]) <= 1e-9 * max(1.0, gd["gnorm_f64/" + key]), key


@pytest.mark.parametrize("what", [A.PGPD_DUAL_CLS, A.PGPD_DUAL_FEAT, A.PGPD_DUAL_STN])
@pytest.mark.parametrize("training", [False, True])
def test_dual_emulator_forward(what, training):
    B, N, k = 5, 37, 3
    st = sub_state(W.make_state(21, k=k, style="wild", dual=True), what)
    x = dual_clouds(22, B, N)
    if what == A.PGPD_DUAL_STN:
        x = x[:, :3]
    ro, rt, _, rsd = port_run(st, x, what, training)
    out, trans, _, est = emu_run(st, x, what, training, k)
    assert np.abs(trans - rt).max() < 2e-5
    if ro is not None:
        assert np.abs(out - ro).max() < (1e-4 if what == A.PGPD_DUAL_CLS else 2e-4)
        if what == A.PGPD_DUAL_CLS:
            assert (out.argmax(1) == ro.argmax(1)).all()
    if training:       # running statistics, updated in place like nn.BatchNorm1d
        for key in A.dual_buffer_keys(what):
            r = rsd[key].numpy()
            if key.endswith("num_batches_tracked"):
                assert int(est[key].reshape(-1)[0]) == int(r) == 1
            else:
                assert np.abs(est[key] - r).max() < 1e-5 * max(1.0, np.abs(r).max()), key


@pytest.mark.parametrize("what,B,N", [(A.PGPD_DUAL_CLS, 6, 45), (A.PGPD_DUAL_FEAT, 4, 70), (A.PGPD_DUAL_STN, 7, 33)])
def test_dual_emulator_backward(what, B, N):
    k = 2
    st = sub_state(W.make_state(31, k=k, style="wild", dual=True), what)
    x = dual_clouds(32, B, N)
    if what == A.PGPD_DUAL_STN:
        x = x[:, :3]
    width = {A.PGPD_DUAL_CLS: k, A.PGPD_DUAL_FEAT: 1024, A.PGPD_DUAL_STN: 1}[what]
    wo, wt = W.normal(33, (B, width)), W.normal(34, (B, 3, 3))
    _, _, rg, _ = port_run(st, x, what, True, wo, wt)
    _, _, rg32, _ = port_run(st, x, what, True, wo, wt, dtype=torch.float32)
    _, _, g, _ = emu_run(st, x, what, True, k, wo, wt)
    for key in A.dual_param_keys(what):
        r = rg[key]
        if key.endswith(".bias") and (".conv" in "." + key or ".fc1" in "." + key or ".fc2" in "." + key):
            # a bias feeding a train-mode BatchNorm: the gradient is identically zero (torch returns rounding noise)
            assert np.abs(g[key]).max() == 0.0, key
            continue
        # judged against the reference's own fp32 error (arg-max routing makes fp32 gradients discontinuous)
        budget = max(5e-4, 20 * rel(rg32[key], r))
        assert rel(g[key], r) < budget, (key, rel(g[key], r), budget)


def _module_for(what, N, k):
    from pointnetgpd_b200.model.pointnet import DualPointNetCls
    full = DualPointNetCls(N, 6, k)
    return {A.PGPD_DUAL_CLS: full, A.PGPD_DUAL_FEAT: full.feat, A.PGPD_DUAL_STN: full.feat.stn1}[what], full


def test_dual_modules_through_the_autograd_glue_on_the_emulator(monkeypatch):
    """The nn.Module classes + torch.autograd glue, with host tensors and the emulator build standing in for libpgpd."""
    from pointnetgpd_b200 import functional as Fn
    monkeypatch.setattr(A, "load", emu_lib)
    B, N, k = 4, 29, 2
    st = W.make_state(51, k=k, style="wild", dual=True)
    x = dual_clouds(52, B, N)
    wo, wt = W.normal(53, (B, k)), W.normal(54, (B, 3, 3))
    mod, _ = _module_for(A.PGPD_DUAL_CLS, N, k)
    mod.load_state_dict({kk: torch.tensor(v) for kk, v in st.items()})
    mod.train()
    pk, bk = Fn._dual_keys(A.PGPD_DUAL_CLS)
    params = [Fn._resolve(mod, key) for key in pk]
    bufs = [Fn._resolve(mod, key) for key in bk]
    logp, trans = Fn._DualFn.apply(A.PGPD_DUAL_CLS, True, k, torch.tensor(x), *params, *bufs)
    ((logp * torch.tensor(wo, dtype=torch.float32)).sum() + (trans * torch.tensor(wt, dtype=torch.float32)).sum()).backward()
    ro, rt, rg, rsd = port_run(st, x, A.PGPD_DUAL_CLS, True, wo, wt)
    assert np.abs(logp.detach().numpy() - ro).max() < 1e-4
    assert rel(mod.feat.conv3.weight.grad.numpy(), rg["feat.conv3.weight"]) < 2e-3
    assert rel(mod.feat.stn2.fc3.weight.grad.numpy(), rg["feat.stn2.fc3.weight"]) < 2e-3
    assert int(mod.feat.stn1.bn1.num_batches_tracked) == 1
    assert np.abs(mod.feat.bn3.running_var.numpy() - rsd["feat.bn3.running_var"].numpy()).max() < 1e-4


@pytest.mark.gpu
@pytest.mark.parametrize("what,B,N,k", [(A.PGPD_DUAL_CLS, 6, 72, 2), (A.PGPD_DUAL_CLS, 32, 500, 3), (A.PGPD_DUAL_FEAT, 9, 130, 2),
                                        (A.PGPD_DUAL_STN, 16, 257, 2)])
def test_dual_modules_gpu(what, B, N, k):
    dev = torch.device("cuda:0")
    st_full = W.make_state(61, k=k, style="wild", dual=True)
    st = sub_state(st_full, what)
    x = dual_clouds(62, B, N)
    if what == A.PGPD_DUAL_STN:
        x = x[:, :3]
    width = {A.PGPD_DUAL_CLS: k, A.PGPD_DUAL_FEAT: 1024, A.PGPD_DUAL_STN: 1}[what]
    wo, wt = W.normal(63, (B, width)), W.normal(64, (B, 3, 3))
    mod, _ = _module_for(what, N, k)
    mod.load_state_dict({kk: torch.tensor(v) for kk, v in st.items()})
    mod = mod.to(dev)
    xt = torch.tensor(x, device=dev)
    # eval
    mod.eval()
    with torch.no_grad():
        res = mod(xt)
    ro, rt, _, _ = port_run(st, x, what, False)
    out, trans = (None, res) if what == A.PGPD_DUAL_STN else res
    assert np.abs(trans.cpu().numpy() - rt).max() < 1e-4
    if out is not None:
        assert np.abs(out.cpu().numpy() - ro).max() < 1e-3
        if what == A.PGPD_DUAL_CLS:
            assert (out.cpu().numpy().argmax(1) == ro.argmax(1)).all()
    # train step of a weighted objective (drives d out and d trans)
    mod.train()
    res = mod(xt)
    out, trans = (None, res) if what == A.PGPD_DUAL_STN else res
    obj = (trans * torch.tensor(wt, dtype=torch.float32, device=dev)).sum()
    if out is not None:
        obj = obj + (out * torch.tensor(wo, dtype=torch.float32, device=dev)).sum()
    obj.backward()
    ro, rt, rg, rsd = port_run(st, x, what, True, wo, wt)
    _, _, rg32, _ = port_run(st, x, what, True, wo, wt, dtype=torch.float32)
    assert np.abs(trans.detach().cpu().numpy() - rt).max() < 1e-4
    if out is not None:
        assert np.abs(out.detach().cpu().numpy() - ro).max() < 1e-3
    for key in A.dual_param_keys(what):
        g = Fn_resolve(mod, key).grad.cpu().numpy()
        r = rg[key]
        if np.linalg.norm(r) < 1e-5:       # analytically zero (biases in front of a train-mode BatchNorm, a T-Net's bn3.bias): fp32 noise
            assert np.abs(g).max() < max(1e-4, 20 * float(np.abs(rg32[key]).max())), key
            continue
        assert rel(g, r) < max(2e-3, 20 * rel(rg32[key], r)), key
    for key in A.dual_buffer_keys(what):
        b = Fn_resolve(mod, key).cpu().numpy()
        r = rsd[key].numpy()
        assert np.abs(b - r).max() < 1e-4 * max(1.0, np.abs(r).max()), key


def Fn_resolve(mod, key):
    from pointnetgpd_b200.functional import _resolve
    return _resolve(mod, key)


@pytest.mark.gpu
def test_dual_golden_gpu():
    """DualPointNetCls on the GPU against numbers written by the unmodified reference class (oracle/make_golden.py)."""
    from pointnetgpd_b200.model.pointnet import DualPointNetCls
    gd = np.load(GOLD)
    B, N, k, seed = [int(v) for v in gd["meta"]]
    st = W.make_state(seed, k=k, style="wild", dual=True)
    x = torch.tensor(dual_clouds(seed + 1000, B, N), device="cuda:0")
    m = DualPointNetCls(N, 6, k)
    m.load_state_dict({kk: torch.tensor(v) for kk, v in st.items()})
    m = m.cuda().eval()
    with torch.no_grad():
        logp, trans = m(x)
    assert np.abs(logp.cpu().numpy() - gd["eval_logp_f64"]).max() < 1e-3
    assert (logp.cpu().numpy().argmax(1) == gd["eval_logp_f64"].argmax(1)).all()
    assert np.abs(trans.cpu().numpy() - gd["eval_trans_f64"]).max() < 1e-4
    m.train()
    logp, trans = m(x)
    wl = torch.tensor(W.normal(seed + 3000, (B, k)), dtype=torch.float32, device="cuda:0")
    wt = torch.tensor(W.normal(seed + 4000, (B, 3, 3)), dtype=torch.float32, device="cuda:0")
    ((logp * wl).sum() + (trans * wt).sum()).backward()
    assert np.abs(logp.detach().cpu().numpy() - gd["train_logp_f64"]).max() < 1e-3
    for name, p in m.named_parameters():
        ref = float(gd["gnorm_f64/" + name])
        if ref < 1e-5:
            continue
        ref32 = float(gd["gnorm_f32/" + name])
        got = float(np.linalg.norm(p.grad.cpu().numpy().astype(np.float64)))
        assert abs(got - ref) < max(5e-3 * ref, 20 * abs(ref32 - ref)), name
    for name, b in m.named_buffers():
        r = gd["buf_f64/" + name]
        assert np.abs(b.cpu().numpy() - r).max() < 1e-4 * max(1.0, np.abs(r).max()), name
