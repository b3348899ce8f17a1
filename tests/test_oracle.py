"""Pin the oracle (torch port + numpy fp64 restatement) to the golden vectors produced by the
UNMODIFIED reference module (oracle/make_golden.py).  CPU only."""
import numpy as np
import pytest
import torch

from oracle import pointnet_np as PN
from oracle import pointnet_torch_port as PT
from golden_util import (CASE_NAMES, SMALL_CASES, load_case, param_names, grad_errors, shipped_state,
                         is_zero_grad_param)


@pytest.mark.parametrize("name", CASE_NAMES)
def test_torch_port_matches_reference_f32(name):
    c = load_case(name)
    g = c["g"]
    sd = PT.to_torch_state(c["state"], torch.float32)
    x = torch.tensor(c["x"])
    with torch.no_grad():
        logp, trans = PT.pointnetcls_forward(sd, x, training=False)
    # same ops, same order, same library -> essentially bit-equal
    assert np.abs(logp.numpy() - g["eval_logp_f32"]).max() < 2e-6
    assert np.abs(trans.numpy() - g["eval_trans_f32"]).max() < 2e-6

    sd = PT.to_torch_state(c["state"], torch.float32, requires_grad=True)
    logp, trans, loss, grads = PT.train_step(sd, x, torch.tensor(c["y"]))
    assert np.abs(logp.numpy() - g["train_logp_f32"]).max() < 1e-5
    assert abs(float(loss) - float(g["train_loss_f32"])) < 1e-6
    errs = grad_errors({k: v.numpy() for k, v in grads.items()}, g, "f32")
    for k, (esub, enorm) in errs.items():
        if is_zero_grad_param(k):
            continue
        assert esub < 1e-3 and enorm < 1e-3, (k, esub, enorm)
    for k, v in sd.items():
        if k.endswith("running_mean") or k.endswith("running_var"):
            assert np.abs(v.numpy() - g["buf_f32/" + k]).max() < 1e-5 * max(1.0, np.abs(g["buf_f32/" + k]).max()), k
        if k.endswith("num_batches_tracked"):
            assert int(v) == int(g["buf_f32/" + k]) == 1


@pytest.mark.parametrize("name", SMALL_CASES)
def test_numpy_fp64_matches_reference_f64(name):
    c = load_case(name)
    g = c["g"]
    sd = PN.cast_state(c["state"], np.float64)
    x = c["x"].astype(np.float64)
    logp_e, trans_e, _, _ = PN.forward(sd, x, training=False)
    assert np.abs(logp_e - g["eval_logp_f64"]).max() < 1e-10
    assert np.abs(trans_e - g["eval_trans_f64"]).max() < 1e-10
    logp, trans, loss, grads, new_stats = PN.nll_train_step(sd, x, c["y"])
    assert np.abs(logp - g["train_logp_f64"]).max() < 1e-9
    assert np.abs(trans - g["train_trans_f64"]).max() < 1e-9
    assert abs(loss - float(g["train_loss_f64"])) < 1e-10
    errs = grad_errors(grads, g, "f64")
    for k, (esub, enorm) in errs.items():
        if is_zero_grad_param(k):
            continue
        assert esub < 1e-7 and enorm < 1e-7, (k, esub, enorm)
    for bn, (rm, rv) in new_stats.items():
        assert np.abs(rm - g["buf_f64/" + bn + ".running_mean"]).max() < 1e-10
        assert np.abs(rv - g["buf_f64/" + bn + ".running_var"]).max() < 1e-10


@pytest.mark.parametrize("name", SMALL_CASES)
def test_numpy_fp64_general_output_grads(name):
    """Second gradient pattern: sum(wl*logp) + sum(wt*trans) -- drives d(trans) too."""
    c = load_case(name)
    g = c["g"]
    sd = PN.cast_state(c["state"], np.float64)
    logp, trans, cache, _ = PN.forward(sd, c["x"].astype(np.float64), training=True)
    grads = PN.backward(sd, cache, c["wl"], c["wt"], training=True)
    errs = grad_errors(grads, g, "f64", prefix="g2")
    for k, (esub, enorm) in errs.items():
        if is_zero_grad_param(k):
            continue
        assert esub < 1e-7 and enorm < 1e-7, (k, esub, enorm)


def test_shipped_checkpoint_known_answer(golden_dir):
    import os
    from oracle import weights as W
    st = shipped_state()
    out = np.load(os.path.join(golden_dir, "shipped_3class_outputs.npz"))
    assert len(st) == 74
    sd = PT.to_torch_state(st, torch.float32)
    for kind, seed in (("box", 123), ("dup", 124)):
        x = torch.tensor(W.make_clouds(seed, 8, 500, kind))
        with torch.no_grad():
            logp, trans = PT.pointnetcls_forward(sd, x, training=False)
        assert np.abs(logp.numpy() - out[f"{kind}_logp_f32"]).max() < 1e-4
        assert (logp.argmax(1).numpy() == out[f"{kind}_logp_f64"].argmax(1)).all()
    # fp64 numpy vs reference fp64
    sd64 = PN.cast_state(st, np.float64)
    x = W.make_clouds(123, 8, 500, "box").astype(np.float64)
    logp, trans, _, _ = PN.forward(sd64, x, training=False)
    assert np.abs(logp - out["box_logp_f64"]).max() < 1e-8


def test_crop_oracle_matches_reference_collect_pc(golden_dir):
    """oracle/grasp_crop_np.py vs golden vectors produced by executing the reference's own collect_pc."""
    import os
    from oracle import grasp_crop_np as OC
    g = np.load(os.path.join(golden_dir, "collect_pc.npz"))
    pc, grasps, T = g["pc"], g["grasps"], g["transform"]
    for i in range(len(grasps)):
        idx, pts = OC.crop(pc, grasps[i], T)
        assert np.array_equal(idx, g[f"in_ind_{i}"]), i
        if len(idx):
            assert np.abs(pts - g[f"pc_t_{i}"]).max() < 1e-15
