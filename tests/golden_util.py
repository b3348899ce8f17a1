"""Helpers shared by the parity tests: load a golden case, rebuild its inputs from the
recipe (oracle.weights), compare gradient summaries."""
import os

import numpy as np

from oracle import weights as W
from oracle.make_golden import sub_idx, CASES, load_shipped_state

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
CASE_NAMES = [c[0] for c in CASES]
SMALL_CASES = [c[0] for c in CASES if c[1] * c[2] <= 2000]


def load_case(name):
    g = np.load(os.path.join(GOLDEN, name + ".npz"))
    B, N, k, seed = [int(v) for v in g["meta"]]
    style, kind = str(g["style"]), str(g["kind"])
    state = W.make_state(seed, k=k, style=style)
    x = W.make_clouds(seed + 1000, B, N, kind)
    y = W.make_labels(seed + 2000, B, k)
    wl = W.normal(seed + 3000, (B, k))
    wt = W.normal(seed + 4000, (B, 3, 3))
    return dict(g=g, B=B, N=N, k=k, seed=seed, state=state, x=x, y=y, wl=wl, wt=wt)


def shipped_state():
    """The 74-entry state dict of the shipped 3-class checkpoint, as reduced in tests/golden (oracle/make_golden.py)."""
    return load_shipped_state(os.path.join(GOLDEN, "shipped_3class_state.npz"))


def param_names(state):
    return [k for k in state if not (k.endswith("running_mean") or k.endswith("running_var")
                                     or k.endswith("num_batches_tracked"))]


# gradients that are analytically zero (SURVEY.md Appendix A): the reference returns ~1e-6 noise
def is_zero_grad_param(name):
    if name.endswith(".bias") and (".conv" in name or name.startswith("conv")):
        return True
    if name.endswith("fc1.bias") or name.endswith("fc2.bias"):
        return True
    if name in ("feat.bn3.bias", "feat.stn.bn3.bias"):
        return True
    return False


def grad_errors(grads, g, tag, prefix="g"):
    """Relative errors of `grads` (name -> array) vs golden summaries: returns
    {name: (rel err of subsample, rel err of norm)} using the golden norm as the scale."""
    out = {}
    for name, arr in grads.items():
        ref_norm = float(g[f"{prefix}norm_{tag}/{name}"])
        ref_sub = g[f"{prefix}sub_{tag}/{name}"].astype(np.float64)
        flat = np.asarray(arr, dtype=np.float64).reshape(-1)
        sub = flat[sub_idx(flat.size)]
        scale = max(ref_norm, 1e-30) * np.sqrt(max(1, sub.size) / max(1, flat.size))
        out[name] = (float(np.linalg.norm(sub - ref_sub) / max(scale, 1e-30)),
                     float(abs(np.linalg.norm(flat) - ref_norm) / max(ref_norm, 1e-30)))
    return out
