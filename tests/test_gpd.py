"""GPDClassifier (PointNetGPD/model/gpd.py:5-31; SURVEY.md 8f row 4): the CUDA implementation (csrc/gpd.cuh) against the oracle's
torch port -- on the CPU through the SIMT emulator build of libpgpd (C ABI, numpy buffers), on the GPU through the nn.Module.
The port is pinned to the unmodified reference class through the reference-generated fixture tests/golden/gpd_pin.npz."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from emu_util import emu_lib, Guarded
from oracle import gpd_torch_port as G
from pointnetgpd_b200 import _abi as A
from pointnetgpd_b200 import synth as W

PIN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "gpd_pin.npz")


def _inputs(seed, B, Cc):
    x = W.normal(seed, (B, Cc, 60, 60)).astype(np.float32)
    y = W.make_labels(seed + 1, B, 2)
    return x, y


def _oracle(sd, x, y, dtype):
    sdd = {k: v.to(dtype).clone().requires_grad_(True) for k, v in sd.items()}
    logp = G.gpd_forward(sdd, torch.tensor(x).to(dtype))
    loss = torch.nn.functional.nll_loss(logp, torch.tensor(y))
    loss.backward()
    return logp.detach().numpy(), {k: v.grad.numpy() for k, v in sdd.items()}


def test_gpd_port_matches_reference():
    """Against what the unmodified reference GPDClassifier computed in eval mode on the same inputs (oracle/make_golden.py)."""
    gd = np.load(PIN)
    for Cc in (3, 12):
        sd = G.make_gpd_state(5, Cc)
        x = torch.tensor(_inputs(6, 3, Cc)[0])
        with torch.no_grad():
            assert torch.equal(torch.tensor(gd[f"logp_c{Cc}"]), G.gpd_forward(sd, x))
    assert list(gd["state_keys"]) == list(G.make_gpd_state(1, 3).keys())


@pytest.mark.parametrize("B,Cc", [(3, 3), (2, 12)])
def test_gpd_emulator_forward_backward(B, Cc):
    lib = emu_lib()
    sd = G.make_gpd_state(11, Cc)
    x, y = _inputs(12, B, Cc)
    ref_logp, ref_g = _oracle(sd, x, y, torch.float64)
    st = {k: np.ascontiguousarray(v.numpy()) for k, v in sd.items()}
    grads = {k: np.full(v.shape, np.nan, np.float32) for k, v in st.items()}
    m, g = A.Gpd(), A.GpdGrad()
    for name in A.GPD_LAYERS:
        getattr(m, name).w, getattr(m, name).b = st[name + ".weight"].ctypes.data, st[name + ".bias"].ctypes.data
        getattr(g, name).dw, getattr(g, name).db = grads[name + ".weight"].ctypes.data, grads[name + ".bias"].ctypes.data
    nbytes = lib.pgpd_gpd_workspace_bytes(B, Cc, A.F_SAVE)
    ws = Guarded(nbytes)
    logp = np.full((B, 2), np.nan, np.float32)
    A.check(lib, lib.pgpd_gpd_forward(C.byref(m), x.ctypes.data, B, Cc, A.F_SAVE, logp.ctypes.data, ws.addr, nbytes, None))
    ws.check()
    assert np.abs(logp - ref_logp).max() < 1e-4
    dlogp = np.zeros((B, 2), np.float32)
    dlogp[np.arange(B), y] = -1.0 / B
    A.check(lib, lib.pgpd_gpd_backward(C.byref(m), C.byref(g), x.ctypes.data, B, Cc, A.F_SAVE, dlogp.ctypes.data, ws.addr, nbytes, None))
    ws.check()
    for k in st:
        r = ref_g[k]
        assert np.linalg.norm(grads[k] - r) / max(np.linalg.norm(r), 1e-12) < 1e-3, k


@pytest.mark.gpu
@pytest.mark.parametrize("B,Cc", [(5, 3), (64, 3), (17, 12)])
def test_gpd_module_gpu(B, Cc):
    from pointnetgpd_b200.model.gpd import GPDClassifier
    sd = G.make_gpd_state(21, Cc)
    x, y = _inputs(22, B, Cc)
    ref_logp, ref_g = _oracle(sd, x, y, torch.float64)
    m = GPDClassifier(Cc)
    m.load_state_dict(sd)
    m = m.cuda().train()
    logp = m(torch.tensor(x).cuda())
    torch.nn.functional.nll_loss(logp, torch.tensor(y).cuda()).backward()
    assert np.abs(logp.detach().cpu().numpy() - ref_logp).max() < 1e-3
    assert (logp.detach().cpu().numpy().argmax(1) == ref_logp.argmax(1)).all()
    for k, p in m.named_parameters():
        r = ref_g[k]
        assert np.linalg.norm(p.grad.cpu().numpy() - r) / max(np.linalg.norm(r), 1e-12) < 5e-3, k
    m.eval()
    with torch.no_grad():
        assert torch.allclose(m(torch.tensor(x).cuda()), logp.detach(), atol=1e-6)


@pytest.mark.gpu
def test_gpd_training_loop_and_pickle(tmp_path):
    """main_1v_gpd.py:123-133 shape of use: Adam on model.parameters(); torch.save(model) / torch.load round trip."""
    from pointnetgpd_b200.model.gpd import GPDClassifier
    sd = G.make_gpd_state(41, 3)
    m = GPDClassifier(3)
    m.load_state_dict(sd)
    m = m.cuda().train()
    x = torch.tensor(_inputs(31, 32, 3)[0]).cuda()
    y = torch.tensor(_inputs(31, 32, 3)[1]).cuda()
    opt = torch.optim.SGD(m.parameters(), lr=0.01)
    # the same loop through the oracle's port, executed by eager PyTorch on the GPU in true fp32: the loss trajectories must agree
    # (plain SGD: Adam's 1/sqrt(v) turns rounding noise of near-zero gradients into O(lr) steps)
    rs = {k: v.cuda().clone().requires_grad_(True) for k, v in sd.items()}
    ropt = torch.optim.SGD(list(rs.values()), lr=0.01)
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        losses = []
        for _ in range(6):
            opt.zero_grad()
            loss = torch.nn.functional.nll_loss(m(x), y)
            loss.backward()
            opt.step()
            ropt.zero_grad()
            rloss = torch.nn.functional.nll_loss(G.gpd_forward(rs, x), y)
            rloss.backward()
            ropt.step()
            losses.append(float(loss.detach()))
            assert abs(float(loss.detach()) - float(rloss.detach())) < 1e-3 * max(1.0, abs(float(rloss.detach())))
        assert losses[-1] < losses[0]
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old
    path = str(tmp_path / "gpd.model")
    torch.save(m, path)
    m2 = torch.load(path, weights_only=False)
    with torch.no_grad():
        assert torch.equal(m2.eval()(x), m.eval()(x))
    with pytest.raises(NotImplementedError):
        GPDClassifier(3, dropout=True).cuda().train()(x)
