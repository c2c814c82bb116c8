"""Generate tests/golden/*.npz by running the UNMODIFIED reference model (build container only).

    python tests/golden/make_golden.py

Each file holds: the full reference state_dict ("sd/<key>"), the input x, a target, the
reference prediction and losses.mpjpe values; taps/<name>.npz next to it holds the reference-side
taps (Adj / w1 / w2 / ContextLayer attributes read off the live module exactly as
environment/test.py:146-157 does).  Two files keep each one under 1 MB.
The GPU box has no /root/reference, so these vectors are what pins the oracle there.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
import _reference as R  # noqa: E402
from oracle import cistgcn_oracle as O  # noqa: E402

CASES = [
    # name,                 E,  V, weights, scale, interpretable
    ("e8_v22_default",      8, 22, "W1", "unit", True),
    ("e8_v22_stress",       8, 22, "W2", "unit", True),
    ("e8_v18_default_mm",   8, 18, "W1", "mm",   True),
    ("e16_v22_stress",     16, 22, "W2", "unit", True),
    ("e8_v22_static_adj",   8, 22, "W2", "unit", False),
]
BATCH = 2


def main():
    mp = R.ref_mpjpe()
    for name, E, V, wset, scale, itp in CASES:
        ref = R.build(E, V, seed=0, interpretable=itp)
        sd = {k: v.clone() for k, v in ref.state_dict().items()}
        if wset == "W2":
            O.stress_init_(sd, seed=7)
            ref.load_state_dict(sd)
        cfg = O.OracleConfig(joints=V, input_gcn=[E] * 4)
        x, tgt = O.synth_inputs(BATCH, cfg, seed=123, scale=scale)
        with torch.no_grad():
            pred = ref(x)[0]
        out = {"x": x.numpy(), "target": tgt.numpy(), "pred": pred.numpy(),
               "meta": np.array([E, V, cfg.input_n, cfg.output_n, int(itp)], dtype=np.int64),
               "mpjpe_all": mp(pred, tgt).numpy(), "mpjpe_frames": mp(pred, tgt, reduce_axis=(0, 2)).numpy(),
               "mpjpe_none": mp(pred, tgt, reduce_axis=None).numpy()}
        taps = {}
        blocks = [(f"st_gcnns.{i}", m) for i, m in enumerate(ref.st_gcnns)] + \
                 [(f"st_gcnns_o.{i}", m) for i, m in enumerate(ref.st_gcnns_o)]
        for p, m in blocks:
            taps[f"{p}.w1"] = m.w1.detach().numpy()
            taps[f"{p}.w2"] = m.w2.detach().numpy()
            if itp:
                taps[f"{p}.dsgn.Adj"] = m.dsgn.Adj.detach().numpy()
                taps[f"{p}.tsgn.Adj"] = m.tsgn.Adj.detach().numpy()
        cl = ref.context_layer
        for a in ("joints", "displacements", "seq_joints_n", "seq_joints_dims"):
            taps[f"context_layer.{a}"] = getattr(cl, a).detach().numpy()
        for k, v in sd.items():
            out["sd/" + k] = v.numpy()
        path = os.path.join(HERE, name + ".npz")
        np.savez_compressed(path, **out)
        os.makedirs(os.path.join(HERE, "taps"), exist_ok=True)
        np.savez_compressed(os.path.join(HERE, "taps", name + ".npz"), **taps)
        print(name, "|pred|max", float(pred.abs().max()), os.path.getsize(path) // 1024, "KiB")


if __name__ == "__main__":
    main()
