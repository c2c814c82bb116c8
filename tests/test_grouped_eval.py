"""Grouped evaluation: per-group per-frame sums in one pass (csrc/eval_grouped.cu: cistgcn_mpjpe_grouped_f32,
cistgcn_eval_metrics_grouped_f32), the module's forward_mpjpe / rollout_mpjpe with `groups`, EvalMetrics with
`n_groups` and horizons past 32 frames, and dist.sharded_eval_grouped.

CPU: the kernels on the SIMT emulator (tests/emu) against the ungrouped kernel and a float64 torch restatement, both
accumulator paths (shared memory / global atomics), out-of-range ids with poison guard bands around the outputs, error
paths, argument checks and the gloo all-reduce at world size 2.  GPU (-m gpu): the nvcc-built library through the module
and EvalMetrics."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from cistgcn_b200 import CISTGCN, _cabi
from cistgcn_b200.metrics import METRICS, EvalMetrics, source_map
from cistgcn_b200.synth import make_opt, synth_inputs

GOLD = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "aux", "eval_metrics.npz"))
M = len(METRICS)
VEL = METRICS.index("velocity")
BONE = METRICS.index("bone_length")
PA = METRICS.index("pa_mpjpe")
ACC_SMEM_DOUBLES = 48 * 1024 // 8       # kAccSmemBytes of csrc/eval_grouped.cu
MAX_CHUNK = 32768                       # CISTGCN_MAX_CHUNK of csrc/cistgcn_api.cu
DEV = "cuda:0"
PAD = 16
POISON_F, POISON_I = 1234.5, -7777


# ----------------------------------------------------------------------------------------------------- references
def golden(device="cpu"):
    tgt = torch.from_numpy(GOLD["target"]).to(device)
    pred = torch.from_numpy(GOLD["pred22"]).to(device)
    w = torch.from_numpy(GOLD["weights"]).to(device)
    smap = source_map(tgt.shape[2], GOLD["dim_used"].tolist(), GOLD["rep32"].tolist(), GOLD["rep22"].tolist()).to(device)
    bones = torch.from_numpy(GOLD["bones"]).to(torch.int32).to(device).contiguous()
    return pred, tgt, w, smap, bones


def synth_metrics_inputs(B, To, seed=0, device="cpu"):
    """Golden skeleton geometry with a longer horizon: target (B, To, 32, 3) and pred (B, To, 22, 3) near it."""
    g = torch.Generator().manual_seed(seed)
    tgt = torch.randn(B, 1, 32, 3, generator=g) + 0.05 * torch.randn(B, To, 32, 3, generator=g).cumsum(1)
    dim_used = torch.from_numpy(GOLD["dim_used"])
    pred = tgt[:, :, dim_used] + 0.1 * torch.randn(B, To, 22, 3, generator=g)
    w = torch.rand(B, To, 32, generator=g)
    _, _, _, smap, bones = golden()
    return pred.contiguous().to(device), tgt.contiguous().to(device), w.to(device), smap.to(device), bones.to(device)


def restate(pred, tgt, smap, bones, w0=None, w1=None):
    """float64 torch restatement of the seven metrics of eval_metrics_kernel: (M, B, To) per-sample sums over joints
    (velocity 0 at the last frame, weighted terms 0 without weights)."""
    T = tgt.double().cpu()
    P = T.clone()
    m = smap.long().cpu()
    used = m >= 0
    P[:, :, used] = pred.double().cpu()[:, :, m[used]]
    B, To = T.shape[:2]
    out = torch.zeros(M, B, To, dtype=torch.float64)
    e = (P - T).norm(dim=-1)
    out[METRICS.index("mpjpe")] = e.sum(-1)
    for k, w in ((METRICS.index("weighted0"), w0), (METRICS.index("weighted1"), w1)):
        if w is not None:
            out[k] = (w.double().cpu() * e).sum(-1)
    scale = (T * P).sum((2, 3)) / (P * P).sum((2, 3))
    out[METRICS.index("n_mpjpe")] = (scale[..., None, None] * P - T).norm(dim=-1).sum(-1)
    out[VEL, :, :-1] = ((P[:, 1:] - P[:, :-1]) - (T[:, 1:] - T[:, :-1])).norm(dim=-1).sum(-1)
    b0, b1 = bones.long().cpu().T
    out[BONE] = ((P[:, :, b0] - P[:, :, b1]).norm(dim=-1) - (T[:, :, b0] - T[:, :, b1]).norm(dim=-1)).abs().sum(-1)
    muX, muY = T.mean(2, keepdim=True), P.mean(2, keepdim=True)
    X0, Y0 = T - muX, P - muY
    X0 = torch.where(X0 ** 2 < 1e-6, torch.full_like(X0, 1e-3), X0)
    nX = X0.pow(2).sum((2, 3)).sqrt().clamp(min=1e-3)
    nY = Y0.pow(2).sum((2, 3)).sqrt()
    H = (X0 / nX[..., None, None]).transpose(-1, -2) @ (Y0 / nY[..., None, None])
    U, s, Vt = torch.linalg.svd(H)
    R = Vt.transpose(-1, -2) @ U.transpose(-1, -2)
    sg = torch.sign(torch.linalg.det(R))
    R[..., 2, :] *= sg[..., None]
    a = (s[..., 0] + s[..., 1] + sg * s[..., 2]) * nX / nY
    t = muX - a[..., None, None] * (muY @ R)
    out[PA] = ((a[..., None, None] * (P @ R) + t) - T).norm(dim=-1).sum(-1)
    return out


def by_group(per_sample, groups, G):
    """(..., B, T) per-sample values -> (G, ..., T) sums per group (ids outside [0, G) dropped)."""
    x = per_sample.movedim(-2, 0)
    keep = (groups >= 0) & (groups < G)
    out = torch.zeros((G,) + x.shape[1:], dtype=torch.float64)
    return out.index_add_(0, groups[keep].long(), x[keep].double())


def assert_metric_sums(got, ref, what=""):
    """got / ref (G, M, To): pa_mpjpe at 2e-4 of its largest value (SVD conditioning), every other metric at 2e-5."""
    for i, name in enumerate(METRICS):
        scale = max(float(ref[:, i].abs().max()), 1e-30)
        tol = (2e-4 if i == PA else 2e-5) * scale
        err = float((got[:, i] - ref[:, i]).abs().max())
        assert err <= tol, (what, name, err, tol)


# ----------------------------------------------------------------------------------------------------- emulator drivers
def guarded(n, dtype):
    """(buffer with PAD poison entries on each side, body view of n zeros)."""
    poison = POISON_F if dtype == torch.float64 else POISON_I
    buf = torch.full((n + 2 * PAD,), poison, dtype=dtype)
    buf[PAD:PAD + n] = 0
    return buf, buf[PAD:PAD + n]


def assert_guards(buf):
    poison = POISON_F if buf.dtype == torch.float64 else POISON_I
    assert (buf[:PAD] == poison).all() and (buf[-PAD:] == poison).all()


def emu_metrics_grouped(L, pred, tgt, smap, bones, G, groups=None, w0=None, assembled=None):
    B, To, Vu, _ = pred.shape
    Vf = tgt.shape[2]
    sbuf, sums = guarded(G * M * To, torch.float64)
    cbuf, counts = guarded(G, torch.int64)
    gi = groups.to(torch.int32).contiguous() if groups is not None else None
    rc = L.cistgcn_eval_metrics_grouped_f32(pred.data_ptr(), tgt.data_ptr(), gi.data_ptr() if gi is not None else None, G,
                                            smap.data_ptr(), bones.data_ptr(), bones.shape[0],
                                            w0.data_ptr() if w0 is not None else None, None,
                                            assembled.data_ptr() if assembled is not None else None,
                                            sums.data_ptr(), counts.data_ptr(), B, To, Vu, Vf, None)
    _cabi.check(rc, "cistgcn_eval_metrics_grouped_f32[emu]", L)
    assert_guards(sbuf)
    assert_guards(cbuf)
    return sums.view(G, M, To), counts


def emu_metrics(L, pred, tgt, smap, bones, w0=None, assembled=None):
    B, To, Vu, _ = pred.shape
    sums = torch.zeros(M, To, dtype=torch.float64)
    rc = L.cistgcn_eval_metrics_f32(pred.data_ptr(), tgt.data_ptr(), smap.data_ptr(), bones.data_ptr(), bones.shape[0],
                                    w0.data_ptr() if w0 is not None else None, None,
                                    assembled.data_ptr() if assembled is not None else None, sums.data_ptr(), B, To, Vu,
                                    tgt.shape[2], None)
    _cabi.check(rc, "cistgcn_eval_metrics_f32[emu]", L)
    return sums


def emu_mpjpe_grouped(L, pred, tgt, G, groups=None):
    B, T, V, _ = pred.shape
    sbuf, sums = guarded(G * T, torch.float64)
    cbuf, counts = guarded(G, torch.int64)
    gi = groups.to(torch.int32).contiguous() if groups is not None else None
    rc = L.cistgcn_mpjpe_grouped_f32(pred.data_ptr(), tgt.data_ptr(), gi.data_ptr() if gi is not None else None, G, B, T, V,
                                     sums.data_ptr(), counts.data_ptr(), None)
    _cabi.check(rc, "cistgcn_mpjpe_grouped_f32[emu]", L)
    assert_guards(sbuf)
    assert_guards(cbuf)
    return sums.view(G, T), counts


@pytest.fixture(scope="module")
def emu():
    import _emu
    return _emu.lib()


# ----------------------------------------------------------------------------------------------------- CPU: metrics kernel
def test_grouped_metrics_match_ungrouped_kernel_on_each_subset(emu):
    pred, tgt, w, smap, bones = golden()
    B, To = tgt.shape[:2]
    groups = torch.arange(B) % 3
    G = 3
    assert G * M * To + G <= ACC_SMEM_DOUBLES                   # shared-memory accumulator
    asm = torch.empty_like(tgt)
    sums, counts = emu_metrics_grouped(emu, pred, tgt, smap, bones, G, groups, w0=w, assembled=asm)
    asm_ref = torch.empty_like(tgt)
    full = emu_metrics(emu, pred, tgt, smap, bones, w0=w, assembled=asm_ref)
    assert torch.equal(asm, asm_ref) and torch.equal(asm, torch.from_numpy(GOLD["assembled"]))
    assert counts.tolist() == [int((groups == g).sum()) for g in range(G)]
    for g in range(G):
        sel = groups == g
        sub = emu_metrics(emu, pred[sel].contiguous(), tgt[sel].contiguous(), smap, bones, w0=w[sel].contiguous())
        assert torch.allclose(sums[g], sub, rtol=1e-12, atol=0), g
    assert torch.allclose(sums.sum(0), full, rtol=1e-12, atol=0)


def test_one_group_and_null_groups_give_the_ungrouped_result(emu):
    pred, tgt, w, smap, bones = golden()
    full = emu_metrics(emu, pred, tgt, smap, bones, w0=w)
    for groups in (None, torch.zeros(tgt.shape[0], dtype=torch.int32)):
        sums, counts = emu_metrics_grouped(emu, pred, tgt, smap, bones, 1, groups, w0=w)
        assert counts.tolist() == [tgt.shape[0]]
        assert torch.allclose(sums[0], full, rtol=1e-12, atol=0)


def test_grouped_metrics_global_accumulator_path(emu):
    """G = 64 at To = 25 does not fit the shared-memory budget: the same sums through global atomics."""
    pred, tgt, w, smap, bones = golden()
    B, To = tgt.shape[:2]
    G = 64
    assert G * M * To + G > ACC_SMEM_DOUBLES
    groups = torch.tensor([5, 63, 5, 0, 63, 17])
    sums, counts = emu_metrics_grouped(emu, pred, tgt, smap, bones, G, groups, w0=w)
    ref = by_group(restate(pred, tgt, smap, bones, w0=w), groups, G)
    assert counts.tolist() == torch.bincount(groups, minlength=G).tolist()
    assert_metric_sums(sums, ref, "global")
    small, _ = emu_metrics_grouped(emu, pred, tgt, smap, bones, 3, torch.tensor([0, 1, 0, 2, 1, 2]), w0=w)
    assert torch.allclose(sums[[5, 63, 17]].sum(0) + sums[0], small.sum(0), rtol=1e-12, atol=0)


@pytest.mark.parametrize("To,G", [(50, 2), (100, 3), (100, 16)])
def test_grouped_metrics_past_32_frames_match_float64_restatement(emu, To, G):
    """Horizons past the ungrouped kernel's 32 frames and past a 64-frame row; (100, 16) takes the global path."""
    pred, tgt, w, smap, bones = synth_metrics_inputs(4, To, seed=To + G)
    groups = torch.tensor([1, 0, 1, G - 1])
    sums, counts = emu_metrics_grouped(emu, pred, tgt, smap, bones, G, groups, w0=w)
    assert (G * M * To + G <= ACC_SMEM_DOUBLES) == (G < 16)
    ref = by_group(restate(pred, tgt, smap, bones, w0=w), groups, G)
    assert counts.tolist() == torch.bincount(groups, minlength=G).tolist()
    assert float(sums[:, VEL, -1].abs().max()) == 0.0
    assert_metric_sums(sums, ref, f"To={To}")


def test_grouped_metrics_skip_out_of_range_ids(emu):
    pred, tgt, w, smap, bones = golden()
    G = 2
    groups = torch.tensor([0, -1, 1, 2, 1, 0])
    asm = torch.empty_like(tgt)
    sums, counts = emu_metrics_grouped(emu, pred, tgt, smap, bones, G, groups, w0=w, assembled=asm)
    assert counts.tolist() == [2, 2]
    assert torch.equal(asm, torch.from_numpy(GOLD["assembled"]))          # the scatter covers every sample
    keep = (groups >= 0) & (groups < G)
    sub = emu_metrics(emu, pred[keep].contiguous(), tgt[keep].contiguous(), smap, bones, w0=w[keep].contiguous())
    assert torch.allclose(sums.sum(0), sub, rtol=1e-12, atol=0)
    for G in (1, 64):                                                    # both accumulator paths
        sums, counts = emu_metrics_grouped(emu, pred, tgt, smap, bones, G, torch.tensor([-1, G, -5, G + 3, 2**30, -2**31]))
        assert counts.abs().sum() == 0 and sums.abs().sum() == 0


# ----------------------------------------------------------------------------------------------------- CPU: mpjpe kernel
@pytest.mark.parametrize("B,T,V,G", [(7, 25, 22, 3), (5, 400, 22, 64), (6, 50, 18, 15)])
def test_grouped_mpjpe_matches_float64_index_add(emu, B, T, V, G):
    g = torch.Generator().manual_seed(B * T)
    pred, tgt = torch.randn(B, T, V, 3, generator=g), torch.randn(B, T, V, 3, generator=g)
    groups = torch.randint(0, G, (B,), generator=g)
    sums, counts = emu_mpjpe_grouped(emu, pred, tgt, G, groups)
    ref = torch.zeros(G, T, dtype=torch.float64).index_add_(0, groups, (pred.double() - tgt.double()).norm(dim=-1).sum(-1))
    assert counts.tolist() == torch.bincount(groups, minlength=G).tolist()
    assert torch.allclose(sums, ref, rtol=1e-6, atol=1e-9), ("smem" if G * T + G <= ACC_SMEM_DOUBLES else "global")
    # against the ungrouped kernel's frame sums: fp64 reordering only
    fs = torch.zeros(T, dtype=torch.float64)
    _cabi.check(emu.cistgcn_mpjpe_f32(pred.data_ptr(), tgt.data_ptr(), B, T, V, None, fs.data_ptr(), None), "mpjpe", emu)
    assert torch.allclose(sums.sum(0), fs, rtol=1e-12, atol=0)
    one, cnt1 = emu_mpjpe_grouped(emu, pred, tgt, 1)
    assert cnt1.tolist() == [B] and torch.allclose(one[0], fs, rtol=1e-12, atol=0)


def test_grouped_mpjpe_accumulates_and_skips_out_of_range_ids(emu):
    B, T, V = 6, 10, 22
    g = torch.Generator().manual_seed(3)
    pred, tgt = torch.randn(B, T, V, 3, generator=g), torch.randn(B, T, V, 3, generator=g)
    for G in (4, 64 * 32):                                               # shared-memory and global paths
        groups = torch.tensor([0, -1, 3, G, 3, 1], dtype=torch.int32)
        sbuf, sums = guarded(G * T, torch.float64)
        cbuf, counts = guarded(G, torch.int64)
        for _ in range(2):                                               # accumulates into what is there
            rc = emu.cistgcn_mpjpe_grouped_f32(pred.data_ptr(), tgt.data_ptr(), groups.data_ptr(), G, B, T, V,
                                               sums.data_ptr(), counts.data_ptr(), None)
            assert rc == 0
        assert_guards(sbuf)
        assert_guards(cbuf)
        keep = torch.tensor([True, False, True, False, True, True])
        ref = torch.zeros(G, T, dtype=torch.float64).index_add_(
            0, groups[keep].long(), (pred[keep].double() - tgt[keep].double()).norm(dim=-1).sum(-1))
        assert torch.allclose(sums.view(G, T), 2 * ref, rtol=1e-6, atol=1e-9)
        assert counts[:4].tolist() == [2, 2, 0, 4] and int(counts.sum()) == 8


def test_grouped_error_paths(emu):
    L = emu
    pred, tgt, w, smap, bones = golden()
    B, To, Vu, _ = pred.shape
    sums = torch.full((3 * M * To,), 7.0, dtype=torch.float64)
    counts = torch.full((3,), 9, dtype=torch.int64)
    p, t, s, c = pred.data_ptr(), tgt.data_ptr(), sums.data_ptr(), counts.data_ptr()
    sm, bo, nb = smap.data_ptr(), bones.data_ptr(), bones.shape[0]

    def metrics(**kw):
        a = dict(pred=p, target=t, groups=None, G=3, smap=sm, bones=bo, nb=nb, sums=s, counts=c, B=B, To=To, Vu=Vu, Vf=32)
        a.update(kw)
        return L.cistgcn_eval_metrics_grouped_f32(a["pred"], a["target"], a["groups"], a["G"], a["smap"], a["bones"], a["nb"],
                                                  None, None, None, a["sums"], a["counts"], a["B"], a["To"], a["Vu"], a["Vf"],
                                                  None)

    for kw in (dict(pred=None), dict(target=None), dict(sums=None), dict(counts=None), dict(smap=None)):
        assert metrics(**kw) == -1 and b"NULL" in L.cistgcn_last_error()
    for kw in (dict(G=0), dict(G=-3), dict(To=0), dict(Vu=0), dict(Vf=0), dict(Vf=65), dict(B=-1), dict(nb=-1),
               dict(bones=None), dict(G=2**30)):
        assert metrics(**kw) == -1, kw
    assert metrics(B=0) == 0

    def mpjpe(**kw):
        a = dict(pred=p, target=t, groups=None, G=3, B=B, T=To, V=Vu, sums=s, counts=c)
        a.update(kw)
        return L.cistgcn_mpjpe_grouped_f32(a["pred"], a["target"], a["groups"], a["G"], a["B"], a["T"], a["V"], a["sums"],
                                           a["counts"], None)

    for kw in (dict(pred=None), dict(target=None), dict(sums=None), dict(counts=None)):
        assert mpjpe(**kw) == -1 and b"NULL" in L.cistgcn_last_error()
    for kw in (dict(G=0), dict(T=0), dict(V=0), dict(V=-1), dict(B=-1), dict(G=2**30)):
        assert mpjpe(**kw) == -1, kw
    assert mpjpe(B=0) == 0
    assert (sums == 7.0).all() and (counts == 9).all()                   # nothing was written


# ----------------------------------------------------------------------------------------------------- module / front end
@pytest.fixture
def no_library(monkeypatch):
    def refuse():
        raise AssertionError("the library was reached")
    monkeypatch.setattr(_cabi, "lib", refuse)


def small_model(V=22, To=25):
    opt = make_opt(8, V, output_n=To)
    torch.manual_seed(0)
    return CISTGCN(opt.architecture_config, opt.learning_config).eval()


def test_module_group_checks_before_the_library(no_library):
    model = small_model()
    x, tgt = synth_inputs(4, 22)
    ok = torch.tensor([0, 1, 2, 1])
    for fn, t in ((model.forward_mpjpe, tgt), (model.rollout_mpjpe, torch.cat([tgt, tgt], 1))):
        with pytest.raises(ValueError, match="n_groups"):
            fn(x, t, ok)
        for bad in (0, -1, 2.5, True, "3"):
            with pytest.raises(ValueError, match="n_groups"):
                fn(x, t, ok, bad)
        with pytest.raises(ValueError, match="groups"):
            fn(x, t, None, 3)
        for bad in (ok[:3], ok[None], ok.float(), ok.bool(), [0, 1, 2, 1]):
            with pytest.raises(ValueError, match="groups"):
                fn(x, t, bad, 3)
        for bad in (torch.tensor([0, 1, 3, 1]), torch.tensor([0, -1, 2, 1])):
            with pytest.raises(ValueError, match="group ids"):
                fn(x, t, bad, 3)
        with pytest.raises(ValueError, match="CUDA"):                    # valid groups: on to the input checks
            fn(x, t, ok.to(torch.int16), 3)
    with pytest.raises(ValueError, match="target"):
        model.forward_mpjpe(x, tgt[:2], ok, 3)
    with pytest.raises(ValueError, match="target"):
        model.rollout_mpjpe(x, tgt.double(), ok, 3)
    model.train()
    with pytest.raises(ValueError, match="eval mode"):
        model.rollout_mpjpe(x, tgt, ok, 3)


def test_eval_metrics_checks_before_the_library(no_library):
    pred, tgt, w, smap, bones = golden()
    for bad in (0, -2, 1.5, True):
        with pytest.raises(ValueError, match="n_groups"):
            EvalMetrics(25, smap, bones.tolist(), device="cpu", n_groups=bad)
    ev = EvalMetrics(25, smap, bones.tolist(), device="cpu", n_groups=3)
    assert ev.counts.shape == (3,) and ev.counts.dtype == torch.int64
    for bad in (torch.zeros(5, dtype=torch.int64), torch.zeros(6), torch.tensor([0, 1, 2, 3, 0, 0]),
                torch.tensor([0, 1, 2, -1, 0, 0])):
        with pytest.raises(ValueError, match="group"):
            ev.compute(pred, tgt, groups=bad)
    with pytest.raises(ValueError, match="CUDA"):
        ev.compute(pred, tgt, groups=torch.tensor([0, 1, 2, 2, 0, 0]))
    ev.count = 6                                                         # six samples passed, none counted
    with pytest.raises(ValueError, match="outside"):
        ev.values()
    with pytest.raises(ValueError, match="outside"):
        ev.values_by_group()


def test_eval_metrics_values_by_group_from_sums():
    pred, tgt, w, smap, bones = golden()
    ev = EvalMetrics(25, smap, bones.tolist(), device="cpu", n_groups=3)
    per = restate(pred, tgt, smap, bones)
    groups = torch.tensor([0, 0, 2, 0, 2, 2])
    ev.group_sums.copy_(by_group(per, groups, 3))
    ev.counts.copy_(torch.tensor([3, 0, 3]))
    ev.count = 6
    vals, byg = ev.values(), ev.values_by_group()
    assert byg["velocity"].shape == (3, 24) and byg["mpjpe"].shape == (3, 25) and vals["velocity"].shape == (24,)
    assert torch.isnan(byg["mpjpe"][1]).all() and torch.isfinite(byg["mpjpe"][[0, 2]]).all()
    ref = per.sum(1) / (6 * 32)
    assert torch.allclose(vals["mpjpe"].double(), ref[0], rtol=1e-6)
    assert torch.allclose(byg["bone_length"][0].double(), per[BONE, groups == 0].sum(0) / (3 * bones.shape[0]), rtol=1e-6)


# ----------------------------------------------------------------------------------------------------- gloo, world size 2
def _worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from cistgcn_b200.dist import sharded_eval_grouped
    B, T, V, G = 7, 12, 22, 4
    g = torch.Generator().manual_seed(5)
    x = torch.randn(B, 10, V, 3, generator=g)
    tgt = torch.randn(B, T, V, 3, generator=g)
    groups = torch.tensor([3, 0, 3, 1, 0, 3, 0])                         # group 2 empty
    pred_all = tgt + 0.1 * x[:, -1:]

    def fn(xs, ts, gs, n):                                               # what forward_mpjpe(x, t, groups, n) returns
        ps = ts + 0.1 * xs[:, -1:]
        e = (ps.double() - ts.double()).norm(dim=-1).sum(-1)
        keep = (gs >= 0) & (gs < n)                                      # the kernel skips ids outside [0, n)
        return ps, torch.zeros(n, T, dtype=torch.float64).index_add_(0, gs[keep], e[keep]), \
            torch.bincount(gs[keep], minlength=n)

    pred, (lo, hi), per, counts = sharded_eval_grouped(fn, x, tgt, groups, G)
    e = (pred_all.double() - tgt.double()).norm(dim=-1).sum(-1)
    ref = torch.zeros(G, T, dtype=torch.float64).index_add_(0, groups, e) / (torch.bincount(groups, minlength=G)[:, None] * V)
    ok = torch.equal(pred, pred_all[lo:hi]) and counts.tolist() == [3, 1, 0, 3]
    ok &= torch.allclose(per[[0, 1, 3]], ref[[0, 1, 3]], rtol=1e-12) and bool(torch.isnan(per[2]).all())
    try:
        sharded_eval_grouped(fn, x, tgt, torch.where(groups == 1, 5, groups), G)
        ok = False
    except ValueError:
        pass
    # EvalMetrics.all_reduce: rank-dependent accumulators, one collective
    _, _, _, smap, bones = golden()
    ev = EvalMetrics(12, smap, bones.tolist(), device="cpu", n_groups=G)
    ev.group_sums.fill_(rank + 1.0)
    ev.counts.copy_(torch.tensor([rank, 1, 0, 2]))
    ev.count = rank + 3
    ev.all_reduce()
    ok &= bool((ev.group_sums == 3.0).all()) and ev.counts.tolist() == [1, 2, 0, 4] and ev.count == 7
    out[rank] = (bool(ok), lo, hi)
    dist.destroy_process_group()


def test_sharded_eval_grouped_and_all_reduce_world2_gloo():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_worker, args=(2, port, out), nprocs=2, join=True)
    assert out[0] == (True, 0, 4) and out[1] == (True, 4, 7)


# ----------------------------------------------------------------------------------------------------- GPU
def gpu_model(E, V, To, dtype="f32"):
    model = small_model(V, To) if E == 8 else None
    if model is None:
        opt = make_opt(E, V, output_n=To)
        torch.manual_seed(0)
        model = CISTGCN(opt.architecture_config, opt.learning_config).eval()
    model = model.to(DEV)
    if dtype == "bf16":
        model.act_dtype = torch.bfloat16
    return model


def frame_sums_by_group(pred, tgt, groups, G):
    e = (pred.double() - tgt.double()).norm(dim=-1).sum(-1).cpu()
    return torch.zeros(G, pred.shape[1], dtype=torch.float64).index_add_(0, groups.cpu().long(), e)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", ["f32", "bf16"])
@pytest.mark.parametrize("V", [22, 18])
@pytest.mark.parametrize("To", [25, 10])
def test_forward_mpjpe_grouped_gpu(dtype, V, To):
    model = gpu_model(32, V, To, dtype)
    B, G = 300, 5
    x, tgt = synth_inputs(B, V, output_n=To)
    x, tgt = x.to(DEV), tgt.to(DEV)
    groups = (torch.arange(B, device=DEV) * 7) % G
    with torch.no_grad():
        ref = model(x)[0]
        pred, sums, counts = model.forward_mpjpe(x, tgt, groups, G)
        pred_cpu_ids, sums_c, counts_c = model.forward_mpjpe(x, tgt, groups.cpu(), G)
        loop = [model.forward_mpjpe(x[groups == g], tgt[groups == g])[1] for g in range(G)]
    assert torch.equal(pred, ref) and torch.equal(pred_cpu_ids, ref)
    assert sums.shape == (G, To) and sums.dtype == torch.float64 and counts.dtype == torch.int64
    assert counts.tolist() == torch.bincount(groups, minlength=G).tolist()
    assert torch.allclose(sums, sums_c, rtol=1e-12, atol=0) and torch.equal(counts, counts_c)
    assert torch.allclose(sums.cpu(), frame_sums_by_group(pred, tgt, groups, G), rtol=1e-6)
    assert torch.allclose(sums, torch.stack(loop), rtol=1e-5)
    _, whole = model.forward_mpjpe(x, tgt)
    assert torch.allclose(sums.sum(0), whole, rtol=1e-5)


@pytest.mark.gpu
def test_forward_mpjpe_grouped_across_chunks_gpu():
    model = gpu_model(32, 22, 25)
    B, G = MAX_CHUNK + 17, 15
    base_x, base_t = synth_inputs(512, 22)
    idx = torch.arange(B) % 512
    x, tgt = base_x[idx].contiguous().to(DEV), base_t[idx].contiguous().to(DEV)
    groups = torch.randint(0, G, (B,), generator=torch.Generator().manual_seed(1))
    with torch.no_grad():
        ref = model(x)[0]
        pred, sums, counts = model.forward_mpjpe(x, tgt, groups, G)
    assert torch.equal(pred, ref)
    assert counts.tolist() == torch.bincount(groups, minlength=G).tolist()
    assert torch.allclose(sums.cpu(), frame_sums_by_group(pred, tgt, groups, G), rtol=1e-6)


@pytest.mark.gpu
@pytest.mark.parametrize("To,H", [(25, 50), (10, 25)])
def test_rollout_mpjpe_grouped_gpu(To, H):
    model = gpu_model(32, 22, To)
    B, G = 200, 4
    x, tgt = synth_inputs(B, 22, output_n=H)
    x, tgt = x.to(DEV), tgt.to(DEV)
    groups = torch.arange(B, device=DEV) % G
    with torch.no_grad():
        ref = model.rollout(x, H)
        pred, sums, counts = model.rollout_mpjpe(x, tgt, groups, G)
        loop = [model.rollout_mpjpe(x[groups == g], tgt[groups == g])[1] for g in range(G)]
    assert torch.equal(pred, ref) and sums.shape == (G, H)
    assert counts.tolist() == [B // G] * G
    assert torch.allclose(sums.cpu(), frame_sums_by_group(pred, tgt, groups, G), rtol=1e-6)
    assert torch.allclose(sums, torch.stack(loop), rtol=1e-5)


@pytest.mark.gpu
def test_grouped_eval_empty_batch_and_empty_groups_gpu():
    model = gpu_model(8, 22, 25)
    x, tgt = synth_inputs(6, 22)
    x, tgt = x.to(DEV), tgt.to(DEV)
    with torch.no_grad():
        pred, sums, counts = model.forward_mpjpe(x[:0], tgt[:0], torch.empty(0, dtype=torch.int64), 3)
        assert pred.shape == (0, 25, 22, 3) and sums.shape == (3, 25) and not sums.any() and not counts.any()
        pred, sums, counts = model.rollout_mpjpe(x[:0], torch.empty(0, 40, 22, 3, device=DEV),
                                                 torch.empty(0, dtype=torch.int32, device=DEV), 2)
        assert pred.shape == (0, 40, 22, 3) and sums.shape == (2, 40) and not counts.any()
        _, sums, counts = model.forward_mpjpe(x, tgt, torch.tensor([0, 0, 2, 2, 2, 0], device=DEV), 4)
    assert counts.tolist() == [3, 0, 3, 0] and not sums[[1, 3]].any()
    pred_m, tgt_m, w, smap, bones = golden(DEV)
    ev = EvalMetrics(25, smap, bones.tolist(), n_groups=4)
    ev.compute(pred_m, tgt_m, groups=torch.tensor([0, 0, 2, 2, 2, 0]))
    byg = ev.values_by_group()
    assert torch.isnan(byg["mpjpe"][[1, 3]]).all() and torch.isfinite(byg["pa_mpjpe"][[0, 2]]).all()
    assert torch.isnan(byg["velocity"][1]).all() and byg["velocity"].shape == (4, 24)
    ev0 = EvalMetrics(25, smap, bones.tolist(), n_groups=2)
    ev0.compute(pred_m[:0], tgt_m[:0], groups=torch.empty(0, dtype=torch.int64))
    assert torch.isnan(ev0.values_by_group()["mpjpe"]).all() and not ev0.values()["mpjpe"].any()
    bad = EvalMetrics(25, smap, bones.tolist(), n_groups=2)
    bad.compute(pred_m, tgt_m, groups=torch.tensor([0, 1, 2, 0, 1, 0], device=DEV))     # id 2: unchecked on the device
    assert bad.counts.tolist() == [3, 2]
    with pytest.raises(ValueError, match="outside"):
        bad.values()


@pytest.mark.gpu
def test_eval_metrics_grouped_to25_gpu():
    pred, tgt, w, smap, bones = golden(DEV)
    groups = torch.tensor([2, 0, 1, 2, 0, 2])
    ev = EvalMetrics(25, smap, bones.tolist(), n_groups=3)
    ev.compute(pred[:4], tgt[:4], weights0=w[:4], groups=groups[:4])
    asm = ev.compute(pred[4:], tgt[4:], weights0=w[4:], groups=groups[4:].to(DEV), want_assembled=True)
    assert torch.equal(asm.cpu(), torch.from_numpy(GOLD["assembled"])[4:])
    pooled = EvalMetrics(25, smap, bones.tolist())
    pooled.compute(pred, tgt, weights0=w)
    vals, ref_vals = ev.values(), pooled.values()
    for name in METRICS:
        assert torch.allclose(vals[name], ref_vals[name], rtol=1e-5, atol=1e-7), name
    byg = ev.values_by_group()
    for gi in range(3):
        sel = (groups == gi).to(DEV)
        one = EvalMetrics(25, smap, bones.tolist())
        one.compute(pred[sel], tgt[sel], weights0=w[sel])
        for name, v in one.values().items():
            assert torch.allclose(byg[name][gi], v, rtol=1e-5, atol=1e-7), (gi, name)
    ref = by_group(restate(pred, tgt, smap, bones, w0=w), groups, 3)
    assert_metric_sums(ev.group_sums.cpu(), ref, "gpu To=25")
    assert torch.equal(ev.counts.cpu(), torch.tensor([2, 1, 3]))


@pytest.mark.gpu
def test_eval_metrics_grouped_on_rollout_to50_gpu():
    """A long-term model rolled out to 50 frames (past the ungrouped kernel's 32), scored per group on the 32-joint
    skeleton of the golden geometry."""
    model = gpu_model(32, 22, 25)
    B, H, G = 96, 50, 3
    x, _ = synth_inputs(B, 22)
    _, tgt32, _, smap, bones = synth_metrics_inputs(B, H, seed=9)
    dim_used = torch.from_numpy(GOLD["dim_used"])
    x = (x + tgt32[:, :1, dim_used]).to(DEV)                            # windows near the targets' first pose
    groups = torch.arange(B) % G
    with torch.no_grad():
        out = model.rollout(x, H)
    ev = EvalMetrics(H, smap, bones.tolist(), n_groups=G)
    ev.compute(out, tgt32.to(DEV), groups=groups)
    assert torch.equal(ev.counts.cpu(), torch.full((G,), B // G))
    ref = by_group(restate(out, tgt32, smap, bones), groups, G)
    assert_metric_sums(ev.group_sums.cpu(), ref, "gpu rollout To=50")
    byg = ev.values_by_group()
    for gi in range(G):
        sel = groups == gi
        one = EvalMetrics(H, smap, bones.tolist())
        one.compute(out[sel.to(DEV)], tgt32[sel].to(DEV))
        for name, v in one.values().items():
            assert torch.allclose(byg[name][gi], v, rtol=1e-5, atol=1e-7), (gi, name)
    assert byg["velocity"].shape == (G, H - 1)
