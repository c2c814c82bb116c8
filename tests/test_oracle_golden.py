"""Pins oracle/cistgcn_oracle.py to the reference module through its golden vectors (eval mode, with taps)."""
import pytest
import torch

import _golden as G
from oracle import cistgcn_oracle as O


@pytest.mark.parametrize("name", G.names())
def test_oracle_matches_golden(name):
    g = G.load(name)
    taps = {}
    itp = g["interpretable"]
    with torch.no_grad():
        pred = O.forward(g["sd"], g["cfg"], g["x"], taps=taps,
                         interpretable_in=[itp] * 5, interpretable_out=[itp])
    assert pred.shape == g["pred"].shape
    assert (pred - g["pred"]).abs().max().item() <= 0.1 * G.tol(g["pred"])
    for k, ref in g["taps"].items():
        got = taps[k]
        assert got.shape == ref.shape, k
        assert (got - ref).abs().max().item() <= 1e-5 * max(1.0, ref.abs().max().item()), k
    assert abs(O.mpjpe(pred, g["target"]).item() - g["mpjpe_all"].item()) <= 1e-3 * max(1, g["pred"].abs().max().item() / 4)
    assert torch.allclose(O.mpjpe(g["pred"], g["target"], (0, 2)), g["mpjpe_frames"], rtol=1e-6, atol=1e-6)
    assert torch.allclose(O.mpjpe(g["pred"], g["target"], None), g["mpjpe_none"], rtol=1e-6, atol=1e-6)
    assert torch.allclose(O.mpjpe(g["pred"], g["target"]), g["mpjpe_all"], rtol=1e-6, atol=1e-6)


def test_feature_quirks():
    """App. E items 1-2: positions leak into the last velocity / acceleration slots."""
    x = torch.randn(2, 10, 5, 3)
    f = O.build_features(x)                        # (B, 10, T, V)
    assert torch.equal(f[:, 0:3].permute(0, 2, 3, 1), x)
    vel = f[:, 6:9].permute(0, 2, 3, 1)
    acc = f[:, 3:6].permute(0, 2, 3, 1)
    assert torch.equal(vel[:, -1], x[:, -1])
    assert torch.equal(acc[:, -1], x[:, -1])
    assert torch.allclose(acc[:, -2], x[:, -1] - (x[:, -1] - x[:, -2]), atol=1e-6)
    assert torch.allclose(f[:, 9], vel.norm(dim=-1), atol=1e-6)


def test_stats_unbiased():
    x = torch.randn(3, 4, 10, 22)
    s = O.get_stats(x)
    assert s.shape == (3, 22)
    assert torch.allclose(s[:, 11], x.reshape(3, 4, -1).std(-1, unbiased=True).std(1, unbiased=True))
