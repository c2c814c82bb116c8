"""Autoregressive rollout past output_n (CISTGCN.rollout / rollout_mpjpe, cistgcn_rollout_f32 / _bf16).

Semantics: K = ceil(H / To) forwards; w_0 = x, p_k = forward(w_k), w_{k+1} = the last Tin frames of cat(w_k, p_k),
out = cat(p_0, ..., p_{K-1})[:, :H].  The rollout must be bit-identical to that loop written with the forward at the
same batch size, match the same loop over the oracle within the fp32 / bf16 bounds of test_gpu_parity.py /
test_bf16_forward.py, and its fused frame sums must be the per-frame MPJPE of its output.
CPU: the SIMT-emulator build (tests/emu) at E = 8.  GPU (-m gpu): the nvcc-built library through the module."""
import dataclasses
import functools
import math

import pytest
import torch

import _golden as G
from cistgcn_b200 import CISTGCN, _cabi
from cistgcn_b200.pack import pack_state_dict
from cistgcn_b200.synth import make_opt
from oracle import cistgcn_oracle as O

DEV = "cuda:0"
TIN = 10
MAX_CHUNK = 32768          # CISTGCN_MAX_CHUNK of csrc/cistgcn_api.cu


def build(E, V, To, weights="W1", seed=0):
    """(model in eval mode on CPU, state_dict clone, OracleConfig)."""
    opt = make_opt(E, V, output_n=To)
    torch.manual_seed(seed)
    m = CISTGCN(opt.architecture_config, opt.learning_config).eval()
    sd = {k: v.clone() for k, v in m.state_dict().items()}
    if weights == "W2":
        O.stress_init_(sd, seed=7)
        m.load_state_dict(sd)
    elif weights != "W1":
        raise ValueError(weights)
    return m, sd, O.OracleConfig(output_n=To, joints=V, input_gcn=[E] * 4)


def inputs(B, cfg, H, scale="unit"):
    """x (B, Tin, V, 3) and a target of H frames."""
    return O.synth_inputs(B, dataclasses.replace(cfg, output_n=H), scale=scale)


def loop(step, x, To, H):
    """The rollout written out: `step` maps a window (B, Tin, V, 3) to a prediction (B, To, V, 3)."""
    w, preds = x, []
    for _ in range(math.ceil(H / To)):
        p = step(w)
        preds.append(p)
        w = torch.cat([w, p], 1)[:, -TIN:].contiguous()
    return torch.cat(preds, 1)[:, :H]


def oracle_loop(sd, cfg, x, H):
    with torch.no_grad():
        return loop(lambda w: O.forward(sd, cfg, w), x, cfg.output_n, H)


def _scale(ref):
    return max(1.0, ref.abs().max().item() / 4)


def _frame_sums(out, tgt):
    return torch.linalg.vector_norm(out.double() - tgt.double(), dim=-1).sum((0, 2))


# ----------------------------------------------------------------------------------------------------- CPU (emulator)
def emu_forward(L, pk, x):
    B, g = x.shape[0], pk.geometry
    pred = torch.empty(B, g.output_n, g.joints, 3)
    ws = torch.empty(L.cistgcn_workspace_bytes(pk.plan_c, B), dtype=torch.uint8)
    rc = L.cistgcn_forward_f32(pk.plan_c, len(pk.plan), pk.blob.data_ptr(), x.data_ptr(), pred.data_ptr(), None, None,
                               ws.data_ptr(), ws.numel(), B, None, None)
    _cabi.check(rc, "cistgcn_forward_f32[emu]", L)
    return pred


def emu_rollout(L, pk, x, H, target=None, sums=True, ws_bytes=None, fill=float("nan")):
    """(rc, out, frame_sums) of cistgcn_rollout_f32; out starts as `fill` everywhere."""
    B, g = x.shape[0], pk.geometry
    out = torch.full((B, max(H, 1), g.joints, 3), fill)
    fs = torch.zeros(max(H, 1), dtype=torch.float64) if sums and target is not None else None
    if ws_bytes is None:
        ws_bytes = L.cistgcn_rollout_workspace_bytes(pk.plan_c, B)
    ws = torch.empty(ws_bytes, dtype=torch.uint8)
    rc = L.cistgcn_rollout_f32(pk.plan_c, len(pk.plan), pk.blob.data_ptr(), x.data_ptr(), H, out.data_ptr(),
                               target.data_ptr() if target is not None else None, fs.data_ptr() if fs is not None else None,
                               ws.data_ptr(), ws.numel(), B, None)
    return rc, out, fs


EMU_B = 2
# An emulated forward costs seconds, so two cases share the horizons of the list between them: 1, To - 3, To, To + 7 and
# 25 (output_n = 10) or 50 (output_n = 25), each joint count, horizon and weight set once.  The full (V, output_n) grid
# runs on the GPU (test_rollout_bitwise_equals_forward_loop_gpu).
EMU_CASES = [(22, 10, "W2", (1, 7, 10, 17, 25)), (18, 25, "W1", (1, 22, 25, 32, 50))]


@functools.lru_cache(maxsize=None)
def emu_case(V, To, weights):
    """Per case, for its longest horizon: inputs, packed weights, the forward loop on the emulator and the oracle loop.
    A window never depends on the horizon, so every shorter horizon is a prefix of these."""
    import _emu
    model, sd, cfg = build(8, V, To, weights)
    H = max(h for v, t, w, hs in EMU_CASES if (v, t, w) == (V, To, weights) for h in hs)
    x, tgt = inputs(EMU_B, cfg, H)
    pk = pack_state_dict(sd, model.geometry(), "cpu")
    L = _emu.lib()
    fwd = loop(lambda w: emu_forward(L, pk, w), x, To, H)
    return L, pk, x, tgt, fwd, oracle_loop(sd, cfg, x, H)


@pytest.mark.parametrize("V,To,weights,H", [(v, t, w, h) for v, t, w, hs in EMU_CASES for h in hs])
def test_emulated_rollout_matches_forward_loop_and_oracle(V, To, weights, H):
    L, pk, x, tgt_all, fwd, ref = emu_case(V, To, weights)
    fwd, ref, tgt = fwd[:, :H], ref[:, :H], tgt_all[:, :H].contiguous()
    assert torch.isfinite(ref).all()
    rc, out, sums = emu_rollout(L, pk, x, H, tgt)
    _cabi.check(rc, "cistgcn_rollout_f32[emu]", L)
    assert out.shape == (EMU_B, H, V, 3) and sums.shape == (H,)
    assert torch.equal(out, fwd)
    assert (out - ref).abs().max().item() <= G.tol(ref)
    assert torch.allclose(sums, _frame_sums(out, tgt), rtol=1e-6, atol=1e-9)
    s = _scale(ref)
    assert abs((sums.sum() / (EMU_B * H * V)).item() - O.mpjpe(ref, tgt).item()) <= 1e-3 * s
    assert torch.allclose((sums / (EMU_B * V)).float(), O.mpjpe(ref, tgt, (0, 2)), rtol=1e-5, atol=1e-3 * s)


def test_emulated_rollout_error_paths():
    L, pk, x, tgt, _, _ = emu_case(22, 10, "W2")
    H = 25
    rc, out, _ = emu_rollout(L, pk, x, 0)
    assert rc == -1 and b"horizon" in L.cistgcn_last_error()
    rc, out, _ = emu_rollout(L, pk, x, H, tgt, sums=False)
    assert rc == -1 and b"together" in L.cistgcn_last_error()
    assert torch.isnan(out).all()
    need = L.cistgcn_rollout_workspace_bytes(pk.plan_c, EMU_B)
    assert need > L.cistgcn_workspace_bytes(pk.plan_c, EMU_B)
    rc, out, _ = emu_rollout(L, pk, x, H, ws_bytes=need - 1)
    assert rc == -1 and b"workspace" in L.cistgcn_last_error()
    assert torch.isnan(out).all()


def test_emulated_rollout_unsupported_shape_writes_nothing():
    """A horizon with no compiled output block fails in the forward's own launcher (-2, same message) before the first
    rollout step writes anything: out keeps its sentinel, frame_sums stay zero."""
    import _emu
    model, sd, cfg = build(8, 22, 15)
    x, tgt = inputs(1, cfg, 20)
    pk = pack_state_dict(sd, model.geometry(), "cpu")
    L = _emu.lib()
    rc, out, sums = emu_rollout(L, pk, x, 20, tgt)
    assert rc == -2
    msg = L.cistgcn_last_error().decode()
    assert "(22, 15)" in msg and "(22,10)" in msg, msg
    assert torch.isnan(out).all()
    assert torch.equal(sums, torch.zeros(20, dtype=torch.float64))


# ----------------------------------------------------------------------------------------------------- module contract
@pytest.fixture
def no_library(monkeypatch):
    def refuse():
        raise AssertionError("the library was reached")
    monkeypatch.setattr(_cabi, "lib", refuse)


def test_rollout_argument_checks_before_the_library(no_library):
    model, _, cfg = build(8, 22, 10)
    x, tgt = inputs(3, cfg, 25)
    for bad in (0, -1, 2.5, True, "3", None):
        with pytest.raises(ValueError, match="horizon"):
            model.rollout(x, bad)
    with pytest.raises(ValueError, match="target"):
        model.rollout_mpjpe(x, tgt[:2])
    with pytest.raises(ValueError, match="target"):
        model.rollout_mpjpe(x, tgt[:, :, :18])
    with pytest.raises(ValueError, match="target"):
        model.rollout_mpjpe(x, tgt.double())
    with pytest.raises(ValueError, match="target"):
        model.rollout_mpjpe(x, tgt[0])
    with pytest.raises(ValueError, match="CUDA"):            # the forward's input checks
        model.rollout(x, 25)


def test_rollout_refuses_train_mode_and_input_gradients(no_library):
    model, _, cfg = build(8, 22, 10)
    x, tgt = inputs(3, cfg, 25)
    model.train()
    with pytest.raises(ValueError, match="eval mode"):
        model.rollout(x, 25)
    with pytest.raises(ValueError, match="eval mode"):
        model.rollout_mpjpe(x, tgt)
    model.eval()
    xg = x.clone().requires_grad_()
    with pytest.raises(ValueError, match="not differentiable"):
        model.rollout(xg, 25)
    with torch.no_grad(), pytest.raises(ValueError, match="CUDA"):     # no grad mode: past that check
        model.rollout(xg, 25)


# ----------------------------------------------------------------------------------------------------- GPU
def forward_loop(model, x, H):
    return loop(lambda w: model(w)[0], x, model.n_output, H)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", ["f32", "bf16"])
@pytest.mark.parametrize("E", [8, 32, 64])
@pytest.mark.parametrize("V", [22, 18])
@pytest.mark.parametrize("To", [10, 25])
def test_rollout_bitwise_equals_forward_loop_gpu(dtype, E, V, To):
    model, _, cfg = build(E, V, To)      # default weights: stress weights do not always survive their own predictions
    B, H = 64, 2 * To + 7
    x, tgt = inputs(B, cfg, H)
    model = model.to(DEV)
    if dtype == "bf16":
        model.act_dtype = torch.bfloat16
    x, tgt = x.to(DEV), tgt.to(DEV)
    with torch.no_grad():
        ref = forward_loop(model, x, H)
        out = model.rollout(x, H)
        out_m, sums = model.rollout_mpjpe(x, tgt)
    assert out.shape == (B, H, V, 3) and torch.isfinite(out).all()
    assert torch.equal(out, ref)
    assert torch.equal(out_m, ref)
    from cistgcn_b200.losses import mpjpe
    assert sums.dtype == torch.float64 and sums.shape == (H,)
    assert torch.allclose(sums, mpjpe(out, tgt, reduce_axis=(0, 2)).double() * (B * V), rtol=1e-6, atol=1e-6)


@pytest.mark.gpu
def test_rollout_across_chunks_gpu():
    """CISTGCN_MAX_CHUNK + 17 samples: the second chunk runs its own K steps on the same window / step buffers."""
    model, _, cfg = build(32, 22, 10)
    B, H = MAX_CHUNK + 17, 25
    base, _ = inputs(512, cfg, H)
    x = base[torch.arange(B) % 512].contiguous().to(DEV)
    model = model.to(DEV)
    with torch.no_grad():
        ref = forward_loop(model, x, H)
        out = model.rollout(x, H)
    assert torch.isfinite(out).all() and torch.equal(out, ref)
    assert torch.equal(out[MAX_CHUNK:MAX_CHUNK + 17], out[MAX_CHUNK % 512:MAX_CHUNK % 512 + 17])


@pytest.mark.gpu
def test_rollout_honours_flags_repacking_and_leaves_taps_gpu():
    model, _, cfg = build(8, 18, 10)
    x, _ = inputs(16, cfg, 27)
    x = x.to(DEV)
    model = model.to(DEV).enable_taps()
    with torch.no_grad():
        model(x)
        taps = model.last_taps
        model.enable_taps(False)
        model.kernel_flags = _cabi.FLAG_FPN_FP32 | _cabi.FLAG_DSTD_MIX_FFMA
        assert torch.equal(model.rollout(x, 27), forward_loop(model, x, 27))
        model.kernel_flags = 0
        before = model.rollout(x, 27)
        p = getattr(model.context_layer.fmap_t, "0").weight
        p.mul_(1.5)                                           # visible to the version counters: re-packed
        after = model.rollout(x, 27)
        assert not torch.equal(before, after)
        assert torch.equal(after, forward_loop(model, x, 27))
        empty, sums = model.rollout_mpjpe(x[:0], torch.empty(0, 27, 18, 3, device=DEV))
    assert model.last_taps is taps
    assert empty.shape == (0, 27, 18, 3) and torch.equal(sums.cpu(), torch.zeros(27, dtype=torch.float64))


@pytest.mark.gpu
# mm-scale inputs with default weights only, as in test_short_horizon.py.  Stress-initialised models do not always survive
# their own prediction as input (at 25 frames step 0 reaches |p| ~ 10-64 and step 1 overflows fp32 in the oracle too), so
# stress weights appear in the one case whose rollout stays finite.
@pytest.mark.parametrize("E,V,To,weights,scale", [
    (8, 22, 10, "W2", "unit"), (32, 22, 10, "W1", "unit"), (32, 18, 10, "W1", "mm"),
    (64, 18, 10, "W1", "unit"), (8, 18, 25, "W1", "unit"), (32, 22, 25, "W1", "mm"), (64, 22, 25, "W1", "unit"),
    (64, 18, 25, "W1", "mm"),
])
def test_rollout_matches_oracle_loop_gpu(E, V, To, weights, scale):
    model, sd, cfg = build(E, V, To, weights)
    B, H = 48, 25 if To == 10 else 50
    x, tgt = inputs(B, cfg, H, scale)
    ref = oracle_loop(sd, cfg, x, H)
    model = model.to(DEV)
    with torch.no_grad():
        out, sums = model.rollout_mpjpe(x.to(DEV), tgt.to(DEV))
    out = out.cpu()
    assert torch.isfinite(out).all()
    assert (out - ref).abs().max().item() <= G.tol(ref)
    s = _scale(ref)
    assert abs((sums.sum() / (B * H * V)).item() - O.mpjpe(ref, tgt).item()) <= 1e-3 * s
    assert torch.allclose((sums / (B * V)).float().cpu(), O.mpjpe(ref, tgt, (0, 2)), rtol=1e-5, atol=1e-3 * s)


@pytest.mark.gpu
@pytest.mark.parametrize("E,V,To", [(32, 22, 10), (64, 18, 25)])
def test_bf16_rollout_matches_oracle_loop_gpu(E, V, To):
    model, sd, cfg = build(E, V, To, "W1")
    B, H = 64, 25 if To == 10 else 50
    x, tgt = inputs(B, cfg, H)
    ref = oracle_loop(sd, cfg, x, H)
    model = model.to(DEV)
    model.act_dtype = torch.bfloat16
    with torch.no_grad():
        out, sums = model.rollout_mpjpe(x.to(DEV), tgt.to(DEV))
    out = out.cpu()
    assert torch.isfinite(out).all()
    assert (out - ref).abs().max().item() <= 3e-2
    assert abs((sums.sum() / (B * H * V)).item() - O.mpjpe(ref, tgt).item()) <= 5e-3


@pytest.mark.gpu
def test_sharded_eval_of_rollout_gpu():
    from cistgcn_b200.dist import sharded_eval_mpjpe
    model, _, cfg = build(32, 22, 10, "W1")
    B, H = 96, 25
    x, tgt = inputs(B, cfg, H)
    x, tgt = x.to(DEV), tgt.to(DEV)
    model = model.to(DEV)
    with torch.no_grad():
        out, sums = model.rollout_mpjpe(x, tgt)
        pred, (lo, hi), m_all, m_frames = sharded_eval_mpjpe(model.rollout_mpjpe, x, tgt, rank=0, world=1)
    assert (lo, hi) == (0, B)
    assert torch.equal(pred, out)
    assert m_frames.shape == (H,)
    assert torch.allclose(m_frames, sums / (B * 22), rtol=1e-12, atol=0)
    assert torch.allclose(m_all, (sums / (B * 22)).mean(), rtol=1e-12, atol=0)
