"""The differentiable path (cistgcn_b200/train.py over csrc/train_ops.cu) against the reference's own autograd:
train-mode forward (batch-statistics BatchNorm, running-stat updates), losses.mpjpe with reduce_axis=[], backward
(every parameter's gradient), Adam; and the eval-mode input gradient.

The reference side is _models.OracleModule: the reference model restated by oracle/cistgcn_oracle.py under PyTorch's
autograd and torch.optim.Adam.  The oracle is pinned to the reference module's outputs in eval mode (tests/golden); in
train mode it uses torch's batch-statistics BatchNorm (F.batch_norm, training=True), the function nn.BatchNorm calls.
CPU: the kernels run on the SIMT emulator (tests/emu).  GPU (-m gpu): the same comparison through the nvcc-built
library on larger shapes."""
import pytest
import torch

import _models as M
from cistgcn_b200.train import DiffGraph, FlatParams, Trainer
from oracle import cistgcn_oracle as O


def _log_parity(title, rows):
    """Observed errors per tensor -> gpurun_out/parity_r2_train.log (copied to profiles/ for the record)."""
    import os
    d = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "gpurun_out")
    if not os.path.isdir(d):
        return
    rows = sorted(rows, key=lambda r: -r[1])
    with open(os.path.join(d, "parity_r2_train.log"), "a") as f:
        f.write(f"== {title}: {len(rows)} tensors; worst max-abs/|g|max ours {rows[0][1]:.2e} (reference fp32 {max(r[2] for r in rows):.2e}); "
                f"worst rel-L2 ours {max(r[3] for r in rows):.2e} (reference fp32 {max(r[4] for r in rows):.2e})\n")
        for r in rows[:5]:
            f.write(f"   {r[0]:60s} max-abs/|g|max ours {r[1]:.2e} ref {r[2]:.2e}   rel-L2 ours {r[3]:.2e} ref {r[4]:.2e}\n")


def _reference_step(E, V, sd, x, tgt, train=True, input_grad=False, interp=True, dtype=torch.float32, device="cpu"):
    ref = M.oracle_module(E, V, interp=interp).to(dtype)
    ref.load_state_dict(sd)
    ref = ref.to(device)
    ref.train(train)
    x, tgt = x.to(dtype).to(device), tgt.to(dtype).to(device)
    xr = x.clone().requires_grad_(input_grad)
    pred = ref(xr)[0]
    loss = torch.mean(torch.norm(pred - tgt, 2, dim=-1))           # losses.mpjpe, reduce_axis=[]  (losses.py:57-60)
    loss.backward()
    grads = {n: p.grad.detach().cpu().clone() for n, p in ref.named_parameters() if p.grad is not None}
    return (pred.detach().cpu(), loss.detach().cpu(), grads, {k: v.detach().cpu().clone() for k, v in ref.state_dict().items()},
            (xr.grad.cpu() if input_grad else None))


def _ours(E, V, sd, x, tgt, lib, device="cpu", train=True, input_grad=False, interp=True):
    opt = M.make_opt(E, V, interp)
    opt.learning_config.dropout = 0.0
    from cistgcn_b200 import CISTGCN
    model = CISTGCN(opt.architecture_config, opt.learning_config)
    model.load_state_dict(sd)
    model = model.to(device)
    flat = FlatParams(model)
    g = DiffGraph(model, flat, lib)
    pred = g.forward(x.to(device), training=train, input_grad=input_grad, param_grads=True)
    sums, dpred = g.mpjpe_loss(pred, tgt.to(device))
    dx = g.backward(dpred)
    loss = sums.sum() / (pred.shape[0] * pred.shape[1] * pred.shape[2])
    return pred, loss, g, model, dx


def _ulp_perturbed(t, gen):
    """t with every element moved by a random fraction of one fp32 ulp (|delta| <= 2^-24 |t|): the same problem to
    working precision."""
    if not torch.is_floating_point(t):
        return t.clone()
    return t * (1.0 + (torch.rand(t.shape, generator=gen, dtype=torch.float64) * 2 - 1).to(t.dtype) * 2.0 ** -24)


def _compare(E, V, B, lib, device, interp=True, train=True, input_grad=False, draws=3):
    model0, sd, cfg = M.build(E, V, "W2", interp=interp)
    x, tgt = O.synth_inputs(B, cfg)
    rp, rl, rg, rsd, rdx = _reference_step(E, V, sd, x, tgt, train, input_grad, interp)
    # Truth = the reference step in fp64.  The yardstick is the reference's OWN fp32 noise against that truth, sampled
    # (1 + draws) times: the plain fp32 run and `draws` fp32 runs whose weights and inputs are moved by less than one ulp
    # (the same problem to working precision; a backward-stable evaluation is allowed exactly the answers of such
    # neighbours).  One sample is not a yardstick here: the ~130 scalar PReLU slope gradients are sums of 10^4 .. 10^6
    # products of both signs whose total is orders of magnitude below the terms, and the gate MLPs normalise with
    # BatchNorm1d over a 3 .. 24 sample batch, so the fp32 error of ONE slope varies by more than 10x between two
    # summation orders (observed: 5e-4 in one run, 1e-2 in the next) while every convolution / linear / BatchNorm tensor
    # sits at 1e-5 .. 1e-4.  The per-tensor maximum over the samples is the noise level the bound multiplies.
    tp, tl, tg, _, tdx = _reference_step(E, V, sd, x, tgt, train, input_grad, interp, dtype=torch.float64)
    rel = lambda got, truth: (got.double() - truth).norm().item() / max(truth.norm().item(), 1e-30)
    noise_l2 = {n: rel(gr, tg[n]) for n, gr in rg.items()}
    noise_dx = rel(rdx, tdx) if input_grad else 0.0
    gen = torch.Generator().manual_seed(99)
    samples = [("cpu", True)] * draws
    if str(device).startswith("cuda"):                              # ATen's CUDA kernels: other summation orders, fp32 accumulators
        samples += [(device, False), (device, True)]
    for dev_s, perturb in samples:
        sdp = {k: _ulp_perturbed(v, gen) for k, v in sd.items()} if perturb else sd
        xp = _ulp_perturbed(x, gen) if perturb else x
        _, _, pg, _, pdx = _reference_step(E, V, sdp, xp, tgt, train, input_grad, interp, device=dev_s)
        for n, gr in pg.items():
            noise_l2[n] = max(noise_l2[n], rel(gr, tg[n]))
        if input_grad:
            noise_dx = max(noise_dx, rel(pdx, tdx))
    pred, loss, g, model, dx = _ours(E, V, sd, x, tgt, lib, device, train, input_grad, interp)
    scale = max(1.0, rp.abs().max().item())
    assert (pred.cpu() - rp).abs().max().item() <= 2e-4 * scale
    assert abs(loss.item() - rl.item()) <= 1e-4 * max(1.0, abs(rl.item()))
    # Per parameter tensor, against the fp64 truth.  TIGHT bound:
    #   (1) relative L2 error <= max(10 x the reference's fp32 noise level on that tensor (above), 2e-3), and
    #   (2) max-abs error <= 5e-3 of the tensor's largest entry + 1e-4 of the largest gradient in the model.
    # The network has kinks: ~130 PReLUs switch slope at 0 and the two max-poolings of the ContextLayer
    # (CISTGCN.py:465-466) route a gradient to ONE arg-max element.  Any two fp32 evaluations (the reference on CPU and on
    # CUDA included) put a handful of the ~10^6 activations per sample on different sides of a kink; each such flip changes
    # one element of a backward map by O(|dy|), i.e. one term of the few-hundred-term sums behind a weight-gradient row: a
    # jump of ~1 % on a few entries of whichever tensors sit right behind the flip, independent of eps and different
    # in every run.  So the tight bound must hold for at least 97 % of the tensors, and EVERY tensor must meet the LOOSE
    # bound: (1) with a floor of 5e-2 and (2) with 5e-2 / 1e-3.  A wrong kernel breaks the loose bound (errors of O(1)); a
    # systematically imprecise one breaks the tight bound on whole families of tensors (that is how the fp32 BatchNorm
    # reductions were found: 10 .. 40 x the noise on every tensor behind a 1-channel BatchNorm).
    # gpurun_out/parity_r2_train.log keeps the observed table.
    worst = ("", 0.0)
    gmax = max(gr.abs().max().item() for gr in tg.values())
    rows, outliers = [], []
    for n, gr in rg.items():
        assert n in g.grads, f"no gradient for {n}"
        got = g.grads[n].cpu().double()
        truth = tg[n]
        den = max(truth.abs().max().item(), 1e-30)
        ours_abs, ref_abs = (got - truth).abs().max().item(), (gr.double() - truth).abs().max().item()
        ours_l2, ref_l2 = rel(got, truth), noise_l2[n]
        live = truth.abs().max().item() > 1e-4 * gmax               # tensors whose gradient is 0 in exact arithmetic: (2) only
        if live:
            rows.append((n, ours_abs / den, ref_abs / den, ours_l2, ref_l2))
        if ours_abs / den > worst[1]:
            worst = (n, ours_abs / den)
        if live:
            assert ours_l2 <= max(10 * ref_l2, 5e-2), (n, ours_l2, ref_l2)
        assert ours_abs <= 5e-2 * den + 1e-3 * gmax, (n, ours_abs, ref_abs, den)
        if (live and ours_l2 > max(10 * ref_l2, 2e-3)) or ours_abs > 5e-3 * den + 1e-4 * gmax:
            outliers.append((n, ours_l2, ref_l2, ours_abs / den))
    _log_parity(f"train-grad E={E} V={V} B={B} interp={interp} device={device} ({len(outliers)} of {len(rg)} tensors outside the tight bound)", rows)
    assert len(outliers) <= 0.03 * len(rg), outliers
    if train:                                                       # running statistics updated like torch (momentum 0.1)
        osd = model.state_dict()
        for k, v in rsd.items():
            if k.endswith("running_mean") or k.endswith("running_var"):
                assert torch.allclose(osd[k].cpu(), v, rtol=1e-4, atol=1e-5), k
            if k.endswith("num_batches_tracked"):
                assert int(osd[k]) == int(v), k
    if input_grad:
        l2 = tdx.norm().item()
        ours_l2 = (dx.cpu().double() - tdx).norm().item() / l2
        ours_abs = (dx.cpu().double() - tdx).abs().max().item()
        _log_parity(f"input-grad E={E} V={V} B={B} device={device}", [("d loss / d x", ours_abs / tdx.abs().max().item(),
                    (rdx.double() - tdx).abs().max().item() / tdx.abs().max().item(), ours_l2, noise_dx)])
        assert ours_l2 <= max(10 * noise_dx, 2e-3), (ours_l2, noise_dx)
        assert ours_abs <= 5e-3 * tdx.abs().max().item(), ours_abs
    return worst


def test_train_step_gradients_match_reference_autograd_emulated():
    import _emu
    worst = _compare(8, 22, 3, _emu.lib(), "cpu")
    print("worst relative gradient error", worst)


def test_eval_mode_input_gradient_matches_reference_emulated():
    import _emu
    _compare(8, 18, 2, _emu.lib(), "cpu", train=False, input_grad=True)


@pytest.mark.gpu
@pytest.mark.parametrize("E,V,B,interp", [(8, 22, 16, True), (32, 22, 24, True), (16, 18, 8, True), (8, 22, 6, False)])
def test_train_step_gradients_match_reference_autograd_gpu(E, V, B, interp):
    from cistgcn_b200 import _cabi
    _compare(E, V, B, _cabi.lib(), "cuda:0", interp=interp)


@pytest.mark.gpu
def test_eval_mode_input_gradient_gpu():
    from cistgcn_b200 import _cabi
    _compare(32, 22, 8, _cabi.lib(), "cuda:0", train=False, input_grad=True)


@pytest.mark.gpu
def test_adam_steps_track_torch_optim_adam():
    """Three full steps (forward, loss, backward, fused Adam with L2-in-gradient weight decay) against the reference
    module + torch.optim.Adam (environment/utils.py:53-57): losses and parameters stay together."""
    from cistgcn_b200 import CISTGCN
    E, V, B = 16, 22, 32
    model0, sd, cfg = M.build(E, V, "W2")
    x, tgt = O.synth_inputs(B, cfg)
    ref = M.oracle_module(E, V)
    ref.load_state_dict(sd)
    ref.train()
    LR = 1e-4          # Adam's update is ~lr * sign(g) at first: a small lr keeps the two fp32 trajectories comparable
    opt_ref = torch.optim.Adam(ref.parameters(), lr=LR, weight_decay=1e-4)
    opt = M.make_opt(E, V)
    opt.learning_config.dropout = 0.0
    model = CISTGCN(opt.architecture_config, opt.learning_config)
    model.load_state_dict(sd)
    model = model.to("cuda:0")
    tr = Trainer(model, lr=LR, weight_decay=1e-4)
    xd, td = x.to("cuda:0"), tgt.to("cuda:0")
    for step in range(3):
        opt_ref.zero_grad()
        lr_ = torch.mean(torch.norm(ref(x)[0] - tgt, 2, dim=-1))
        lr_.backward()
        opt_ref.step()
        sums = tr.step(xd, td)
        loss = (sums.sum() / (B * 25 * V)).item()
        assert abs(loss - lr_.item()) <= 2e-3 * max(1.0, abs(lr_.item())), (step, loss, lr_.item())
    worst = 0.0
    for n, p in ref.named_parameters():
        got = dict(model.named_parameters())[n].detach().cpu()
        worst = max(worst, (got - p.detach()).abs().max().item())
    # Adam's first steps move every parameter by ~lr regardless of gradient scale; sign flips of ~0 gradients are the
    # only place the two trajectories can part, so compare in units of lr
    assert worst <= 3 * 2 * LR, worst


@pytest.mark.gpu
def test_reference_style_training_loop_through_autograd():
    """environment/train.py:54-107 verbatim against the drop-in module: model.train(); outputs = model(inputs);
    loss = mpjpe(target, outputs[0]); optimizer.zero_grad(); loss.backward(); optimizer.step() with torch.optim.Adam."""
    from cistgcn_b200 import CISTGCN, mpjpe
    E, V, B = 16, 22, 16
    model0, sd, cfg = M.build(E, V, "W2")
    x, tgt = O.synth_inputs(B, cfg)
    ref = M.oracle_module(E, V)
    ref.load_state_dict(sd)
    ref.train()
    opt_ref = torch.optim.Adam(ref.parameters(), lr=1e-4, weight_decay=1e-4)
    opt = M.make_opt(E, V)
    opt.learning_config.dropout = 0.0
    model = CISTGCN(opt.architecture_config, opt.learning_config)
    model.load_state_dict(sd)
    model = model.to("cuda:0").train()
    optim = torch.optim.Adam(model.parameters(), lr=1e-4, weight_decay=1e-4)
    xd, td = x.to("cuda:0"), tgt.to("cuda:0")
    for step in range(2):
        opt_ref.zero_grad()
        lr_ = torch.mean(torch.norm(ref(x)[0] - tgt, 2, dim=-1))
        lr_.backward()
        outputs = model(xd)
        assert isinstance(outputs, tuple) and len(outputs) == 1
        loss = mpjpe(td, outputs[0])
        optim.zero_grad()
        loss.backward()
        if step == 0:
            gmax = max(p.grad.abs().max().item() for p in ref.parameters())
            for (n, p), q in zip(ref.named_parameters(), model.parameters()):
                assert q.grad is not None, n
                assert (q.grad.cpu() - p.grad).abs().max().item() <= 3e-2 * p.grad.abs().max().item() + 1e-3 * gmax, n   # loose: the
                # tight, noise-anchored comparison is test_train_step_gradients_match_reference_autograd_gpu
        opt_ref.step()
        optim.step()
        assert abs(loss.item() - lr_.item()) <= 2e-3 * max(1.0, abs(lr_.item()))
    # eval after training: the fused inference kernels see the updated weights and running statistics
    model.eval()
    ref.eval()
    with torch.no_grad():
        pe, pr = model(xd)[0].cpu(), ref(x)[0]
    assert (pe - pr).abs().max().item() <= 5e-2 * max(1.0, pr.abs().max().item())


@pytest.mark.gpu
def test_train_mode_dropout_is_active_and_unbiased():
    """learning_config.dropout > 0: two train-mode forwards differ (fresh masks), eval-mode ones do not."""
    from cistgcn_b200 import CISTGCN
    opt = M.make_opt(8, 22)
    opt.learning_config.dropout = 0.1
    torch.manual_seed(0)
    model = CISTGCN(opt.architecture_config, opt.learning_config).to("cuda:0")
    x, _ = O.synth_inputs(8, O.OracleConfig(joints=22, input_gcn=[8] * 4))
    xd = x.to("cuda:0")
    model.train()
    a = model(xd)[0].detach().clone()
    b = model(xd)[0].detach().clone()
    assert torch.isfinite(a).all() and not torch.equal(a, b)
    model.eval()
    with torch.no_grad():
        c, d = model(xd)[0], model(xd)[0]
    assert torch.equal(c, d)


@pytest.mark.gpu
def test_cuda_graph_training_step_matches_eager_launches():
    """Trainer(cuda_graph=True): forward + loss + backward replayed as one captured CUDA graph.  With dropout 0 the replayed
    steps are bit-identical to host-launched ones (same kernels, same order); with dropout on and a frozen optimizer the
    loss still changes from replay to replay (the masks follow the device-side step counter, not a captured constant)."""
    from cistgcn_b200 import CISTGCN
    E, V, B = 16, 22, 32
    x, tgt = O.synth_inputs(B, O.OracleConfig(joints=V, input_gcn=[E] * 4))
    xd, td = x.to("cuda:0"), tgt.to("cuda:0")

    def run(graph, dropout, lr, steps=5):
        opt = M.make_opt(E, V)
        opt.learning_config.dropout = dropout
        torch.manual_seed(0)
        model = CISTGCN(opt.architecture_config, opt.learning_config).to("cuda:0")
        tr = Trainer(model, lr=lr, weight_decay=1e-4 if lr else 0.0, cuda_graph=graph)
        losses = [float(tr.step(xd, td).sum()) for _ in range(steps)]
        return losses, tr.flat.flat.clone(), {k: v.clone() for k, v in model.state_dict().items()}, tr

    le, pe, sde, _ = run(False, 0.0, 1e-3)
    lg, pg, sdg, tr = run(True, 0.0, 1e-3)
    assert tr._cg is not None and tr._cg[4] > 1000                  # captured, and it holds the whole step
    assert le == lg and torch.equal(pe, pg)
    for k in sde:
        assert torch.equal(sde[k], sdg[k]), k                        # running statistics, num_batches_tracked
    ld, _, _, _ = run(True, 0.1, 0.0, steps=6)
    assert len(set(ld[2:])) == len(ld[2:]), ld                       # replays 3..6: fresh masks every time
