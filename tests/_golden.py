"""Helpers to read tests/golden/*.npz and their taps in tests/golden/taps/ (written by tests/golden/make_golden.py)."""
import glob
import os

import numpy as np
import torch

from oracle import cistgcn_oracle as O

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def names():
    return sorted(os.path.splitext(os.path.basename(p))[0] for p in glob.glob(os.path.join(GOLDEN_DIR, "*.npz")))


def load(name):
    d = np.load(os.path.join(GOLDEN_DIR, name + ".npz"))
    E, V, tin, tout, itp = (int(v) for v in d["meta"])
    cfg = O.OracleConfig(input_n=tin, output_n=tout, joints=V, input_gcn=[E] * 4)
    sd = {k[3:]: torch.from_numpy(d[k]) for k in d.files if k.startswith("sd/")}
    t = np.load(os.path.join(GOLDEN_DIR, "taps", name + ".npz"))
    taps = {k: torch.from_numpy(t[k]) for k in t.files}
    g = {k: torch.from_numpy(d[k]) for k in ("x", "target", "pred", "mpjpe_all", "mpjpe_frames", "mpjpe_none")}
    g.update(cfg=cfg, sd=sd, taps=taps, interpretable=bool(itp), embed=E)
    return g


def tol(ref: torch.Tensor, base: float = 1e-4) -> float:
    """fp32 parity bound (SURVEY.md 8c / BASELINE.md section 4): 1e-4 absolute on unit-scale
    outputs, scaled by max(1, |ref|_inf / 4) when the reference output itself is large."""
    return base * max(1.0, float(ref.abs().max()) / 4.0)

