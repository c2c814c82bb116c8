"""Short-term models (output_n = 10, the H3.6M 80-400 ms protocol) on the inference path.

The output block st_gcnns_o sees (T, V) = (joints, output_n), so at 10 frames it runs its own instantiations of the
three-stage DSTD-GC kernels, (22, 10) and (18, 10); the FPN stack runs on the tcgen05 kernel with 2-chunk (K = 16) layers.
CPU: the same sources on the SIMT emulator (tests/emu) against the oracle.  GPU (-m gpu): the nvcc-built library through
the drop-in module.  Bounds as in test_gpu_parity.py / test_bf16_forward.py."""
import types

import pytest
import torch

import _golden as G
from cistgcn_b200 import CISTGCN, _cabi
from cistgcn_b200.pack import F, pack_state_dict
from oracle import cistgcn_oracle as O

TO = 10
DEV = "cuda:0"


def make_opt10(E=8, V=22, interp=True):
    ns = types.SimpleNamespace
    mp = ns(input_n=10, output_n=TO, joints=V, n_txcnn_layers=4, txc_kernel_size=3, reduction=8, hidden_dim=64,
            input_gcn=ns(model_complexity=[E] * 4, interpretable=[interp] * 5),
            output_gcn=ns(model_complexity=[3], interpretable=[interp]), clipping=15)
    return ns(architecture_config=ns(model="CISTGCN_0", model_params=mp), learning_config=ns(dropout=0.1))


def build10(E, V, weights="W1", interp=True, seed=0):
    """(model in eval mode on CPU, state_dict clone, OracleConfig) of a 10-frame model."""
    opt = make_opt10(E, V, interp)
    torch.manual_seed(seed)
    m = CISTGCN(opt.architecture_config, opt.learning_config).eval()
    sd = {k: v.clone() for k, v in m.state_dict().items()}
    if weights == "W2":
        O.stress_init_(sd, seed=7)
        m.load_state_dict(sd)
    elif weights != "W1":
        raise ValueError(weights)
    return m, sd, O.OracleConfig(output_n=TO, joints=V, input_gcn=[E] * 4)


def _oracle(sd, cfg, x, interp=True, taps=None):
    with torch.no_grad():
        return O.forward(sd, cfg, x, taps=taps, interpretable_in=[interp] * 5, interpretable_out=[interp])


def _scale(ref):
    return max(1.0, ref.abs().max().item() / 4)


def _check_taps(got, ref_taps, stress):
    assert got
    for k, t in got.items():
        r = ref_taps[k]
        g = t.cpu().reshape(r.shape)
        err = (g - r).abs().max().item()
        assert err <= 1e-4 * max(1.0, r.abs().max().item()), k
        if stress:
            assert err <= 1e-4 * r.abs().max().item(), (k, err, r.abs().max().item())


def _emu_run(L, pk, x, flags=0, fill=0.0):
    B = x.shape[0]
    g = pk.geometry
    pk.plan_c[F["CP_FLAGS"]] = flags
    pred = torch.full((B, g.output_n, g.joints, 3), fill)
    ws = torch.empty(L.cistgcn_workspace_bytes(pk.plan_c, B), dtype=torch.uint8)
    taps_struct, holders = _cabi.make_taps(g, B, "cpu")
    rc = L.cistgcn_forward_f32(pk.plan_c, len(pk.plan), pk.blob.data_ptr(), x.contiguous().data_ptr(), pred.data_ptr(),
                               None, None, ws.data_ptr(), ws.numel(), B, taps_struct, None)
    return rc, pred, holders


def fpn_tc_supported(pk):
    """Plain-Python statement of what the tcgen05 FPN launcher accepts (csrc/cistgcn_api.cu, fpn_tc_supported)."""
    td = pk.tail_desc()
    fd = pk.fpn_descs()
    To, V, Tin, n = td[F["CT_TOUT"]], td[F["CT_V"]], td[F["CT_TIN"]], pk.geometry.n_fpn
    if To > 25 or Tin > 16 or td[F["CT_F"]] != 10 or V not in (22, 18) or n > 4:
        return False
    for l in range(n):
        f = fd[l * F["CF_COUNT"]: (l + 1) * F["CF_COUNT"]]
        if f[F["CF_TC_KC"]] != (f[F["CF_CIN"]] + 15) // 16 * 2 or f[F["CF_TC_W"]] <= 0 or f[F["CF_TC_PRM"]] <= 0:
            return False
        if f[F["CF_TC_W16"]] <= 0 or (f[F["CF_RESID"]] != 0) != (l > 0):
            return False
    return True


# ----------------------------------------------------------------------------------------------------- CPU (emulator)
@pytest.mark.parametrize("E", [8, 32])
@pytest.mark.parametrize("V", [22, 18])
@pytest.mark.parametrize("weights", ["W1", "W2"])
@pytest.mark.parametrize("interp", [True, False])
def test_emulated_forward_matches_oracle(E, V, weights, interp):
    import _emu
    model, sd, cfg = build10(E, V, weights, interp)
    B = 2
    x, tgt = O.synth_inputs(B, cfg)
    ref_taps = {}
    ref = _oracle(sd, cfg, x, interp, ref_taps)
    pred, sums, taps = _emu.forward(sd, model.geometry(), x, tgt)
    assert pred.shape == (B, TO, V, 3)
    assert (pred - ref).abs().max().item() <= G.tol(ref)
    s = _scale(ref)
    assert abs((sums.sum() / (B * TO * V)).item() - O.mpjpe(ref, tgt).item()) <= 1e-3 * s
    assert torch.allclose((sums / (B * V)).float(), O.mpjpe(ref, tgt, (0, 2)), rtol=1e-5, atol=1e-3 * s)
    if interp:
        assert taps["st_gcnns_o.0.dsgn.Adj"].shape == (B, TO, V, V)
        assert taps["st_gcnns_o.0.tsgn.Adj"].shape == (B, V, TO, TO)
    _check_taps(taps, ref_taps, weights == "W2")


@pytest.mark.parametrize("V", [22, 18])
def test_emulated_flag_twins(V):
    """Every FP32-FMA twin of the three stages (REDUCE_FFMA, ADJ_FFMA, MIX_FFMA) against the default kernels: each within
    the bound of the oracle and of the others.  MIX_FFMA is the tile kernel; the default stage 3 of the 10-frame output
    block is the warp-per-sample kernel, so the two predictions differ in their last bits."""
    import _emu
    model, sd, cfg = build10(8, V, "W2")
    x, _ = O.synth_inputs(2, cfg)
    ref = _oracle(sd, cfg, x)
    L = _emu.lib()
    outs = {}
    for name, flags in (("default", 0), ("reduce", _cabi.FLAG_DSTD_REDUCE_FFMA), ("adj", _cabi.FLAG_DSTD_ADJ_FFMA),
                        ("mix", _cabi.FLAG_DSTD_MIX_FFMA)):
        rc, pred, _ = _emu_run(L, pack_state_dict(sd, model.geometry(), "cpu"), x, flags)
        _cabi.check(rc, f"cistgcn_forward_f32[emu, {name}]", L)
        assert (pred - ref).abs().max().item() <= G.tol(ref), name
        outs[name] = pred
    for a in outs:
        for b in outs:
            assert (outs[a] - outs[b]).abs().max().item() <= G.tol(ref), (a, b)
    assert not torch.equal(outs["default"], outs["mix"])


@pytest.mark.parametrize("V", [22, 18])
@pytest.mark.parametrize("tc", [False, True])
def test_emulated_fused_path_rejects_ten_frame_output_block(V, tc):
    """The round-1 fused kernel is not built for the 10-frame output block: CISTGCN_FLAG_DSTD_FUSED (with or without
    _TC) returns an error naming the shape and writes no prediction."""
    import _emu
    model, sd, cfg = build10(8, V)
    x, _ = O.synth_inputs(2, cfg)
    L = _emu.lib()
    flags = _cabi.FLAG_DSTD_FUSED | (_cabi.FLAG_DSTD_TC if tc else 0)
    rc, pred, _ = _emu_run(L, pack_state_dict(sd, model.geometry(), "cpu"), x, flags, fill=float("nan"))
    assert rc == -2
    msg = L.cistgcn_last_error().decode()
    assert f"(T, V) = ({V}, 10)" in msg, msg
    assert torch.isnan(pred).all()
    # the output block on its own, through the single-block entry point
    pk = pack_state_dict(sd, model.geometry(), "cpu")
    d = pk.block_desc("out", 0)
    xin = torch.randn(2, 3 * V * TO)
    out = torch.full((2, 3 * V * TO), float("nan"))
    rc = L.cistgcn_dstd_block_f32(d, pk.blob.data_ptr(), xin.data_ptr(), out.data_ptr(), 2, None, None, 0, flags, None)
    assert rc == -2 and f"({V}, 10)" in L.cistgcn_last_error().decode()
    assert torch.isnan(out).all()


@pytest.mark.parametrize("V", [22, 18])
@pytest.mark.parametrize("weights", ["W1", "W2"])
def test_pack_reports_tcgen05_fpn_at_ten_frames(V, weights):
    model, sd, _ = build10(8, V, weights)
    pk = pack_state_dict(sd, model.geometry(), "cpu")
    assert pk.fpn_tc and pk.fpn_tc_reason == ""
    assert fpn_tc_supported(pk)
    fd = pk.fpn_descs()
    kcs = [fd[l * F["CF_COUNT"] + F["CF_TC_KC"]] for l in range(pk.geometry.n_fpn)]
    assert kcs == [2, 2, 2, 2]


def test_unsupported_horizon_names_the_built_shapes():
    import _emu
    opt = make_opt10(8, 22)
    opt.architecture_config.model_params.output_n = 15
    torch.manual_seed(0)
    model = CISTGCN(opt.architecture_config, opt.learning_config).eval()
    cfg = O.OracleConfig(output_n=15, joints=22, input_gcn=[8] * 4)
    x, _ = O.synth_inputs(1, cfg)
    L = _emu.lib()
    rc, _, _ = _emu_run(L, pack_state_dict(model.state_dict(), model.geometry(), "cpu"), x)
    assert rc == -2
    msg = L.cistgcn_last_error().decode()
    assert "(22, 15)" in msg and "(22,10)" in msg and "(18,10)" in msg and "(22,25)" in msg, msg


# ----------------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
# mm-scale inputs with default weights only: under stress weights they overflow fp32 in the input blocks of the oracle itself
@pytest.mark.parametrize("E,V,weights,scale", [
    (8, 22, "W1", "unit"), (8, 18, "W2", "unit"), (32, 22, "W1", "unit"), (32, 22, "W1", "mm"), (32, 18, "W1", "mm"),
    (32, 18, "W2", "unit"), (64, 22, "W2", "unit"), (64, 18, "W1", "unit"), (64, 18, "W1", "mm"),
])
def test_forward_matches_oracle_gpu(E, V, weights, scale):
    model, sd, cfg = build10(E, V, weights)
    B = 48
    x, tgt = O.synth_inputs(B, cfg, scale=scale)
    ref_taps = {}
    ref = _oracle(sd, cfg, x, taps=ref_taps)
    model = model.to(DEV).enable_taps()
    with torch.no_grad():
        pred = model(x.to(DEV))[0].cpu()
        pm, sums = model.forward_mpjpe(x.to(DEV), tgt.to(DEV))
    assert pred.shape == (B, TO, V, 3) and torch.isfinite(pred).all()
    assert (pred - ref).abs().max().item() <= G.tol(ref)
    assert torch.equal(pm.cpu(), pred)
    if weights == "W1" and scale == "unit":
        assert (pred - ref).abs().max().item() <= 1e-4
    s = _scale(ref)
    assert abs((sums.sum() / (B * TO * V)).item() - O.mpjpe(ref, tgt).item()) <= 1e-3 * s
    assert torch.allclose((sums / (B * V)).float().cpu(), O.mpjpe(ref, tgt, (0, 2)), rtol=1e-5, atol=1e-3 * s)
    _check_taps(model.last_taps, ref_taps, False)


@pytest.mark.gpu
@pytest.mark.parametrize("E,V", [(32, 22), (16, 18)])
def test_tcgen05_fpn_runs_at_ten_frames(E, V):
    """The default forward runs the FPN stack on tcgen05 (split bf16 + fp16 operands), CISTGCN_FLAG_FPN_FP32 on the FP32-FMA
    kernel: both within the bound, and not bit-equal, so the tensor-core kernel really ran."""
    model, sd, cfg = build10(E, V, "W2")
    x, _ = O.synth_inputs(64, cfg)
    ref = _oracle(sd, cfg, x)
    model = model.to(DEV)
    assert model.pack().fpn_tc
    with torch.no_grad():
        tc = model(x.to(DEV))[0].cpu()
        model.kernel_flags = _cabi.FLAG_FPN_FP32
        ffma = model(x.to(DEV))[0].cpu()
    assert (tc - ref).abs().max().item() <= G.tol(ref)
    assert (ffma - ref).abs().max().item() <= G.tol(ref)
    assert not torch.equal(tc, ffma)
    assert (tc - ffma).abs().max().item() <= G.tol(ref)


@pytest.mark.gpu
@pytest.mark.parametrize("E,V", [(32, 22), (64, 18)])
def test_bf16_forward_at_ten_frames(E, V):
    model, sd, cfg = build10(E, V, "W1")
    B = 64
    x, tgt = O.synth_inputs(B, cfg)
    ref = _oracle(sd, cfg, x)
    model = model.to(DEV)
    with torch.no_grad():
        p32, _ = model.forward_mpjpe(x.to(DEV), tgt.to(DEV))
        model.act_dtype = torch.bfloat16
        p16, s16 = model.forward_mpjpe(x.to(DEV), tgt.to(DEV))
    p32, p16 = p32.cpu(), p16.cpu()
    assert torch.isfinite(p16).all() and not torch.equal(p16, p32)
    assert (p16 - ref).abs().max().item() <= 3e-2
    assert abs((s16.sum() / (B * TO * V)).item() - O.mpjpe(ref, tgt).item()) <= 5e-3


@pytest.mark.gpu
def test_batch_across_chunks_matches_per_sample_results():
    """40 000 samples cross the 32 768-sample chunk: every replica of a sample is bit-identical, the batch equals the
    samples run on their own, and a spot check matches the oracle."""
    model, sd, cfg = build10(32, 22, "W2")
    base, _ = O.synth_inputs(500, cfg)
    B = 40000
    x = base[torch.arange(B) % 500].contiguous().to(DEV)
    model = model.to(DEV)
    with torch.no_grad():
        pred = model(x)[0]
        alone = model(base.to(DEV))[0]
    for k in range(B // 500):
        assert torch.equal(pred[k * 500:(k + 1) * 500], alone), k
    ref = _oracle(sd, cfg, base[:32])
    assert (alone[:32].cpu() - ref).abs().max().item() <= G.tol(ref)


@pytest.mark.gpu
def test_interpretation_attributes_at_ten_frames():
    model, sd, cfg = build10(8, 22, "W2")
    B = 5
    x, _ = O.synth_inputs(B, cfg)
    ref_taps = {}
    _oracle(sd, cfg, x, taps=ref_taps)
    model = model.to(DEV).enable_taps()
    with torch.no_grad():
        model(x.to(DEV))
    shapes = {"st_gcnns_o.0.dsgn.Adj": (B, TO, 22, 22), "st_gcnns_o.0.tsgn.Adj": (B, 22, TO, TO),
              "st_gcnns_o.0.w1": (B, 3), "st_gcnns_o.0.w2": (B, 3), "context_layer.displacements": (B, TO),
              "context_layer.seq_joints_n": (B, TO, 22), "context_layer.seq_joints_dims": (B, 3, TO, 22),
              "st_gcnns.1.dsgn.Adj": (B, 22, 10, 10)}
    for key, shape in shapes.items():
        node = model
        for k in key.split("."):
            node = getattr(node, k)
        assert tuple(node.shape) == shape, key
        ref = ref_taps[key]
        assert (node.cpu().reshape(ref.shape) - ref).abs().max().item() <= 1e-4 * ref.abs().max().item(), key
    out0 = getattr(model.st_gcnns_o, "0")
    assert out0.tsgn.gcn.A is out0.tsgn.Adj and out0.dsgn.gcn.A is out0.dsgn.Adj


@pytest.mark.gpu
def test_sharded_eval_and_metrics_at_ten_frames():
    from cistgcn_b200.dist import sharded_eval_mpjpe
    from cistgcn_b200.metrics import EvalMetrics, source_map
    model, sd, cfg = build10(32, 22, "W1")
    x, tgt = O.synth_inputs(96, cfg)
    ref = _oracle(sd, cfg, x)
    model = model.to(DEV)
    with torch.no_grad():
        pred, (lo, hi), m_all, m_frames = sharded_eval_mpjpe(model.forward_mpjpe, x.to(DEV), tgt.to(DEV), rank=0, world=1)
    assert (lo, hi) == (0, 96)
    assert (pred.cpu() - ref).abs().max().item() <= G.tol(ref)
    assert abs(m_all.item() - O.mpjpe(ref, tgt).item()) <= 1e-3 * _scale(ref)
    assert torch.allclose(m_frames.float().cpu(), O.mpjpe(ref, tgt, (0, 2)), atol=1e-3 * _scale(ref))
    ev = EvalMetrics(TO, source_map(22, list(range(22))))
    ev.compute(pred, tgt.to(DEV))
    vals = ev.values()
    assert vals["mpjpe"].shape == (TO,) and vals["velocity"].shape == (TO - 1,)
    assert torch.allclose(vals["mpjpe"].cpu(), m_frames.float().cpu(), rtol=1e-5, atol=1e-6)


@pytest.mark.gpu
def test_train_step_then_eval_forward_at_ten_frames():
    """One train-mode step (differentiable path, batch-statistics BatchNorm, Adam) of a 10-frame model, then the eval-mode
    inference kernels on the updated weights and running statistics against the oracle on those weights."""
    from cistgcn_b200.train import Trainer
    E, V, B = 16, 22, 32
    opt = make_opt10(E, V)
    opt.learning_config.dropout = 0.0
    torch.manual_seed(0)
    model = CISTGCN(opt.architecture_config, opt.learning_config)
    sd0 = {k: v.clone() for k, v in model.state_dict().items()}
    O.stress_init_(sd0, seed=7)
    model.load_state_dict(sd0)
    cfg = O.OracleConfig(output_n=TO, joints=V, input_gcn=[E] * 4)
    x, tgt = O.synth_inputs(B, cfg)
    model = model.to(DEV)
    tr = Trainer(model, lr=1e-4, weight_decay=1e-4)
    sums = tr.step(x.to(DEV), tgt.to(DEV))
    with torch.no_grad():
        ref_train = O.forward({k: v.clone() for k, v in sd0.items()}, cfg, x, train=True, bn_updates={})
    loss_ref = O.mpjpe(ref_train, tgt).item()
    assert sums.shape == (TO,)
    assert abs(sums.sum().item() / (B * TO * V) - loss_ref) <= 2e-3 * max(1.0, loss_ref)
    model.eval()
    sd1 = {k: v.detach().cpu().clone() for k, v in model.state_dict().items()}
    assert any(not torch.equal(sd1[k], sd0[k]) for k in sd0 if k.endswith(".weight"))
    assert any(not torch.equal(sd1[k], sd0[k]) for k in sd0 if k.endswith("running_mean"))
    with torch.no_grad():
        pred = model(x.to(DEV))[0].cpu()
    ref = _oracle(sd1, cfg, x)
    assert (pred - ref).abs().max().item() <= G.tol(ref)
