"""Drop-in boundary (SURVEY.md 8b): constructor, state_dict layout, init stream, packing."""
import copy

import pytest
import torch

import _golden as G
from cistgcn_b200 import CISTGCN
from cistgcn_b200.pack import F
from _models import make_opt




@pytest.mark.parametrize("name", G.names())
def test_state_dict_layout_matches_golden(name):
    g = G.load(name)
    opt = make_opt(g["embed"], g["cfg"].joints, g["interpretable"])
    m = CISTGCN(opt.architecture_config, opt.learning_config)
    mine = m.state_dict()
    assert list(mine.keys()) == list(g["sd"].keys())
    for k, v in g["sd"].items():
        assert tuple(mine[k].shape) == tuple(v.shape), k
    m.load_state_dict(g["sd"], strict=True)


def test_constructor_does_not_mutate_config():
    opt = make_opt(16)
    before = copy.deepcopy(opt.architecture_config.model_params.input_gcn.model_complexity)
    CISTGCN(opt.architecture_config, opt.learning_config)
    CISTGCN(opt.architecture_config, opt.learning_config)       # the reference raises IndexError here (App. E 9)
    assert opt.architecture_config.model_params.input_gcn.model_complexity == before
    assert CISTGCN.__name__ == "CISTGCN"                         # name-based routing, environment/test.py:98-99


@pytest.mark.parametrize("E,V,interp", [(8, 22, True), (8, 18, True)])
def test_same_seed_same_initial_weights_as_reference(E, V, interp):
    """torch.manual_seed(0) + the constructor draw the reference's initial weights: the default-weight golden files
    store the reference module's own state_dict under that seed (tests/golden/make_golden.py)."""
    ref = G.load({22: "e8_v22_default", 18: "e8_v18_default_mm"}[V])["sd"]
    opt = make_opt(E, V, interp)
    torch.manual_seed(0)
    m = CISTGCN(opt.architecture_config, opt.learning_config)
    ms = m.state_dict()
    assert list(ref.keys()) == list(ms.keys())
    for k in ref:
        assert torch.equal(ref[k], ms[k]), k


def test_pack_plan_layout():
    opt = make_opt(8)
    m = CISTGCN(opt.architecture_config, opt.learning_config).eval()
    pk = m.pack("cpu")
    n = F["CP_HEADER_COUNT"] + 5 * F["CB_COUNT"] + 4 * F["CF_COUNT"] + F["CT_COUNT"] + F["CB_COUNT"]
    assert len(pk.plan) == n
    assert pk.plan[F["CP_WEIGHT_FLOATS"]] == pk.blob.numel()
    assert all(off % 4 == 0 for off in pk.offsets.values())
    b0 = pk.block_desc("in", 0)
    assert b0[F["CB_CI"]] == 10 and b0[F["CB_CO"]] == 8 and b0[F["CB_IN_MODE"]] == 1
    b4 = pk.block_desc("in", 4)
    assert (b4[F["CB_OUT_SC"]], b4[F["CB_OUT_ST"]], b4[F["CB_OUT_SV"]]) == (22, 220, 1)
    bo = pk.block_desc("out", 0)
    assert (bo[F["CB_T"]], bo[F["CB_V"]], bo[F["CB_IN_SC"]], bo[F["CB_IN_ST"]], bo[F["CB_IN_SV"]]) == (22, 25, 1, 3, 66)
    # repack only when something changed
    assert m.pack("cpu") is pk
    with torch.no_grad():
        m.prelus._modules["0"].weight.add_(0.1)
    assert m.pack("cpu") is not pk


def test_forward_rejects_bad_inputs():
    opt = make_opt(8)
    m = CISTGCN(opt.architecture_config, opt.learning_config).eval()
    with pytest.raises(ValueError):
        m(torch.zeros(2, 10, 22, 3))                 # CPU tensor: no fallback
    with pytest.raises(ValueError):
        m(torch.zeros(2, 9, 22, 3))
    with pytest.raises(ValueError):
        m(torch.zeros(2, 10, 22, 3, dtype=torch.float64))


def test_pack_cache_sees_parameter_changes():
    """ADVICE r1: the packed-weight cache must not serve stale weights.  In-place updates through the autograd-visible
    API, storage swaps and replaced Parameter objects are detected by the (data_ptr, version) key; writes through
    `.data` (invisible to PyTorch's version counters) need repack() / invalidate_pack() or check_weights=True."""
    import torch
    import _models as M
    model, sd, cfg = M.build(8, 22, "W2")
    first = model.pack("cpu")
    assert model.pack("cpu") is first                                       # unchanged state: cached
    conv = model.st_gcnns._modules["0"].dsgn.tcn._modules["0"]
    with torch.no_grad():
        conv.weight.mul_(1.5)                                               # bumps _version
    second = model.pack("cpu")
    assert second is not first and not torch.equal(second.blob, first.blob)
    conv.weight = torch.nn.Parameter(conv.weight.detach() * 0.5)            # replaced Parameter object
    third = model.pack("cpu")
    assert third is not second and not torch.equal(third.blob, second.blob)
    conv.weight.data.mul_(2.0)                                              # invisible to the version counter
    assert model.pack("cpu") is third                                       # documented blind spot ...
    fourth = model.repack("cpu")                                            # ... closed by an explicit repack
    assert fourth is not third and not torch.equal(fourth.blob, third.blob)
    model.check_weights = True                                              # or by the checksum mode
    fifth = model.pack("cpu")
    conv.weight.data.mul_(0.5)
    sixth = model.pack("cpu")
    assert sixth is not fifth and not torch.equal(sixth.blob, fifth.blob)
    assert model.pack_count >= 5 and model.last_pack_ms > 0


def test_forward_with_grad_input_raises_clearly():
    import torch
    import _models as M
    model, sd, cfg = M.build(8, 22, "W1")
    x = torch.zeros(1, 10, 22, 3, requires_grad=True)
    with pytest.raises(ValueError):                                # CPU tensor: no CPU fallback (the GPU path differentiates)
        model(x)
