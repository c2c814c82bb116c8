"""Shared model / input builders for the tests."""
import types

import torch

from cistgcn_b200 import CISTGCN
from oracle import cistgcn_oracle as O


def make_opt(E=8, V=22, interp=True):
    ns = types.SimpleNamespace
    mp = ns(input_n=10, output_n=25, joints=V, n_txcnn_layers=4, txc_kernel_size=3, reduction=8, hidden_dim=64,
            input_gcn=ns(model_complexity=[E] * 4, interpretable=[interp] * 5),
            output_gcn=ns(model_complexity=[3], interpretable=[interp]), clipping=15)
    return ns(architecture_config=ns(model="CISTGCN_0", model_params=mp), learning_config=ns(dropout=0.1))


def build(E, V, weights="W1", interp=True, seed=0):
    """(model in eval mode on CPU, state_dict clone, OracleConfig)."""
    opt = make_opt(E, V, interp)
    torch.manual_seed(seed)
    m = CISTGCN(opt.architecture_config, opt.learning_config).eval()
    sd = {k: v.clone() for k, v in m.state_dict().items()}
    if weights == "W2":
        O.stress_init_(sd, seed=7)
        m.load_state_dict(sd)
    elif weights != "W1":
        raise ValueError(weights)
    return m, sd, O.OracleConfig(joints=V, input_gcn=[E] * 4)


class OracleModule(CISTGCN):
    """The reference model as an nn.Module whose forward is oracle/cistgcn_oracle.py on the module's own parameters and
    buffers, run by PyTorch on any device and dtype, with PyTorch autograd for every gradient.  The tests use it where
    they need the reference module itself, which is not part of the repository.  The oracle is pinned to the reference
    module's outputs in eval mode (tests/golden); the parameters come from this package's constructor, whose seeded
    state_dict equals the reference's (test_module_contract).  No dropout: callers set it to 0."""

    def __init__(self, E, V, interp=True):
        opt = make_opt(E, V, interp)
        super().__init__(opt.architecture_config, opt.learning_config)
        self.oracle_cfg = O.OracleConfig(joints=V, input_gcn=[E] * 4)
        self.interp = interp

    def forward(self, x):
        sd = dict(self.named_parameters())
        sd.update(self.named_buffers())
        upd = {}
        pred = O.forward(sd, self.oracle_cfg, x, train=self.training, bn_updates=upd,
                         interpretable_in=[self.interp] * 5, interpretable_out=[self.interp])
        with torch.no_grad():
            for k, v in upd.items():
                sd[k].copy_(v)
            if self.training:
                for k, v in sd.items():
                    if k.endswith("num_batches_tracked"):
                        v += 1
        return (pred,)


def oracle_module(E, V, seed=0, interp=True):
    """OracleModule in eval mode, initialised under torch.manual_seed(seed) like the reference constructor."""
    torch.manual_seed(seed)
    return OracleModule(E, V, interp).eval()
