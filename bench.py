#!/usr/bin/env python
"""bench.py -- sequences/sec of the CIST-GCN hot path (BASELINE.json metric).

    python bench.py [--gpus N --steps K --warmup W]                      # configs[1]: E=32, V=22, batch 65536 / GPU, fp32
    python bench.py --embed 16 | --embed 8 --batch 256                   # configs[1] (E=16) / configs[0] shape on the GPU
    python bench.py --mode mpjpe --embed 64 --joints 18 --batch 262144 --scaling strong --gpus N      # configs[2]
    python bench.py --mode train --batch 128 --gpus 8                    # configs[4]: data-parallel training step
    python bench.py --impl reference ...                                 # the reference's own CPU implementation
    python bench.py ... --dump-outputs DIR                               # also write the last timed step's results

A "step" is one pass of the path over one batch of synthetic sequences.  --mode forward: CISTGCN.forward;
--mode mpjpe: forward + losses.mpjpe (fused per-frame sums; with N > 1 the 208-byte sums are all-reduced over NCCL
inside the timed region and both the `[]` and `(0, 2)` reductions are derived).  N > 1: launched by torchrun, one rank
per GPU.  --scaling weak: every rank owns --batch sequences; strong: --batch is the GLOBAL batch, sharded by rank.
No collective is on the forward's data path.  Prints ONE JSON line.

--dump-outputs DIR writes what the last timed step returned, as DIR/<name>.npy (float32 / float64), so that two builds
can be compared output for output: inputs and weights are seeded, so the same arguments give the same inputs.
forward: pred.npy, the predictions of DUMP_ROWS sequences (a fixed, seeded sample of the batch; all of it when smaller);
mpjpe: mpjpe_all.npy and mpjpe_per_frame.npy; train: frame_sums.npy and parameters.npy (the flat parameter vector after
the step).  With N > 1, rank 0 writes its own results.
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

UNIT = "sequences/s"
FP32_FMA_PEAK_TFLOPS = 148 * 128 * 2 * 1.965e9 / 1e12      # CUDA-core FP32 FMA peak at max SM clock (74.5)
# SURVEY.md 8(d): algorithmic FLOPs / sequence (2*MAC of conv+mm+bmm, measured on the reference)
FLOPS_PER_SEQ = {(22, 8): 37.06e6, (22, 16): 40.45e6, (22, 32): 52.22e6, (22, 64): 95.68e6,
                 (18, 8): 29.59e6, (18, 16): 32.32e6, (18, 32): 41.87e6, (18, 64): 77.26e6}
FPN_FLOPS_PER_SEQ = {22: 29.5e6, 18: 29.5e6 * 18 / 22}
DUMP_ROWS = 4096            # --dump-outputs: sequences of pred kept (4096 x 25 x 22 x 3 fp32 = 27 MB)
DUMP_MAX_BYTES = 64 << 20


def metric_name(V, mode):
    what = {"forward": "forward", "mpjpe": "forward + MPJPE eval", "train": "training step (fwd + bwd + grad all-reduce + Adam)"}[mode]
    shape = "H36M 10->25 frames, 22 joints" if V == 22 else f"AMASS 10->25 frames, {V} joints"
    return f"sequences/sec CIST-GCN {what} ({shape})"


def bytes_per_seq(V, E, s=4):
    """SURVEY.md 8(d): one-kernel-per-block compulsory HBM traffic per sequence."""
    return s * V * (80 * E + 2683)


def stage_bytes_per_seq(E, V, T=10, To=25, act_bytes=4):
    """Compulsory HBM bytes per sequence of every kernel kind of THIS partition (DESIGN.md section 5): each kernel
    reads its inputs once and writes its outputs once, weights amortised over the batch.  Keys = profile kind names.
    act_bytes: storage of the activation tensors between the input blocks and into the FPN (2 in the bf16 forward)."""
    blocks = [(10, E, T, V, True)] + [(E, E, T, V, False)] * 3 + [(E, 10, T, V, False), (3, 3, V, To, False)]
    red = adj = mix = fused = 0
    for i, (ci, co, t, v, raw) in enumerate(blocks):
        ch, cg, tv = ci // 2, max(co // 2, 1), t * v
        ab_in = 4 if (raw or i == 5) else act_bytes
        ab_out = 4 if i == 5 else act_bytes
        x_in = ab_in * (3 * tv if raw else ci * tv)
        rec = 4 * ((2 + 2 * t) + 2 * cg * v + 2 * ch * v + 2 * ch * t)
        aj = 4 * (2 * co + v * t * t + t * v * v)
        red += x_in + rec
        adj += rec + aj
        mix += x_in + aj + ab_out * co * tv
        fused += x_in + ab_out * co * tv
    tv = T * V
    return {"dstd_reduce_kernel": red, "dstd_adj_kernel": adj, "dstd_mix_kernel": mix,
            "dstd_block_kernel": fused, "fpn_kernel": act_bytes * 10 * tv + 4 * 3 * To * V,
            "tail_kernel": 4 * (3 * tv + 3 * 3 * To * V), "mpjpe_kernel": 4 * 2 * 3 * To * V}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def measured_tensor_peak():
    """Dense bf16 TFLOP/s, sustained figure (the FPN kernel is timed inside a long step)."""
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        d = json.load(open(p))
        for k in ("bf16_tflops_sustained", "bf16_tflops"):
            if k in d:
                return float(d[k]), f"measured {k} (MEASURED_PEAKS.json)"
    return 1400.0, "fallback sustained (B200_PROFILING.md)"


def fpn_tc_issued_flops_per_seq():
    """Tensor FLOPs the tcgen05 FPN kernel ISSUES per sequence (csrc/fpn_tc.cuh): per k-step and 128-position tile one
    M128 N96 K16 bf16 MMA + one M128 N32 K16 fp16 MMA; 2 tiles; layer 0 has 1 k-step per tap, layers 1-3 have 2;
    27 taps + 3 compress slices (2 k-steps) per layer."""
    ksteps_tiles = 2 * ((27 * 1 + 3 * 2) + 3 * (27 * 2 + 3 * 2))
    return ksteps_tiles * 2.0 * 128 * (96 + 32) * 16


def _host(t):
    """t on the host as a float32 / float64 numpy array."""
    import torch
    t = t.detach().cpu()
    return (t if t.dtype == torch.float64 else t.float()).numpy()


def _row_sample(t):
    """A fixed, seeded sample of DUMP_ROWS rows of t (sorted indices), or t itself when it has no more rows."""
    import torch
    if t.shape[0] <= DUMP_ROWS:
        return t
    idx = torch.randperm(t.shape[0], generator=torch.Generator().manual_seed(0))[:DUMP_ROWS].sort().values
    return t[idx.to(t.device)]


def write_dump(d, arrays):
    import numpy as np
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_MAX_BYTES:
        raise SystemExit(f"--dump-outputs: {total} bytes exceed {DUMP_MAX_BYTES}")
    os.makedirs(d, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(d, name + ".npy"), a)


class ClockSampler(threading.Thread):
    """Samples SM clock + throttle reasons through `nvidia-smi -lms 200` while the timed region runs."""

    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.proc, self.first = index, [], None, 0

    def mark(self):
        """The timed region starts now: only rows that arrive from here on are reported.  (The process itself is started
        before the warm-up steps: NVML initialisation on a fresh box takes a few hundred ms and must not overlap the timed
        region.)"""
        self.first = len(self.rows)

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                parts = [p.strip() for p in line.split(",")]
                if len(parts) == 6:
                    self.rows.append(parts)
        except Exception:
            pass

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
        self.join(timeout=2)
        rows = self.rows[self.first:] or self.rows
        self.rows = rows
        sm = [int(r[0]) for r in rows if r[0].isdigit()]
        mx = [int(r[1]) for r in rows if r[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[2 + i] == "Active" for r in self.rows)]
        return {"sm_mhz": int(statistics.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(self.rows)}


# ---------------------------------------------------------------------------------------------------------------
# CPU arm: the UNMODIFIED reference module (oracle/_ref, vendored by build(); kind "reference") when it is there,
# otherwise the oracle port (kind "port").  The only places bench.py touches oracle/.
# ---------------------------------------------------------------------------------------------------------------
def _cpu_forward_fn(E, V, mode):
    """(callable(x, target) -> None, kind, description).  Reference module in eval mode under no_grad, fp32
    (train mode: environment/train.py:54-107 -- forward, losses.mpjpe, backward, torch.optim.Adam step)."""
    import torch
    from oracle import ref_loader
    if mode == "train":
        if not ref_loader.available():
            raise SystemExit("bench --mode train needs the reference module for its CPU arm (oracle/_ref, built by build())")
        ref = ref_loader.build(E, V).train()
        optim = torch.optim.Adam(ref.parameters(), lr=0.01, weight_decay=1e-4)      # environment/utils.py:53-57
        def fn(x, tgt):
            optim.zero_grad()
            loss = torch.mean(torch.norm(ref(x)[0] - tgt, 2, dim=-1))
            loss.backward()
            optim.step()
        return fn, "reference", f"unmodified reference CISTGCN module ({ref_loader.which()} copy), train mode, fwd + bwd + torch.optim.Adam"
    if ref_loader.available():
        ref = ref_loader.build(E, V)                              # torch.manual_seed(0) + reference constructor
        def mpjpe(pred, target):                                  # losses.py:57-60 restated (SURVEY.md App. D)
            return torch.mean(torch.norm(pred - target, 2, dim=-1), [])
        def fn(x, tgt):
            with torch.no_grad():
                pred = ref(x)[0]
                if mode == "mpjpe":
                    mpjpe(pred, tgt)
        return fn, "reference", f"unmodified reference CISTGCN module ({ref_loader.which()} copy), eval, no_grad"
    from oracle import cistgcn_oracle as O
    model = _make_model(E, V)
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    cfg = O.OracleConfig(joints=V, input_gcn=[E] * 4)
    def fn(x, tgt):
        with torch.no_grad():
            pred = O.forward(sd, cfg, x)
            if mode == "mpjpe":
                O.mpjpe(pred, tgt)
    return fn, "port", "oracle port of the reference algorithm (reference copy not vendored), eval, no_grad"


def cpu_baseline(E, V, mode, budget_s, batch=256):
    """The reference on this box's host cores, on a bounded sample of the same workload."""
    import torch
    from cistgcn_b200.synth import synth_inputs
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    fn, kind, what = _cpu_forward_fn(E, V, mode)
    x, tgt = synth_inputs(batch, V)
    for _ in range(2):
        fn(x, tgt)
    times, t_end = [], time.time() + budget_s
    while len(times) < 3 or (time.time() < t_end and len(times) < 200):
        t0 = time.perf_counter()
        fn(x, tgt)
        times.append(time.perf_counter() - t0)
    med = statistics.median(times)
    return {"value": batch / med, "unit": UNIT, "cores": cores, "kind": kind,
            "sample": f"{len(times)} passes over batch {batch} (E={E}, V={V}, fp32, {mode}), median; {what}; "
                      f"{torch.get_num_threads()} torch threads"}


def _make_model(E, V):
    import torch
    from cistgcn_b200 import CISTGCN
    from cistgcn_b200.synth import make_opt
    opt = make_opt(E, V)
    torch.manual_seed(0)
    return CISTGCN(opt.architecture_config, opt.learning_config).eval()


def workload_name(args, world):
    E, V = args.embed, args.joints
    shape = f"{'H36M' if V == 22 else 'AMASS'} shape (10 in / 25 out frames, {V} joints x 3)"
    what = {"forward": "forward", "mpjpe": "forward + MPJPE eval",
            "train": "data-parallel training step (train-mode fwd + bwd + one NCCL gradient all-reduce + Adam)"}[args.mode]
    if args.scaling == "strong":
        bs = f"global batch {args.batch} sharded over {world} GPU(s)"
    else:
        bs = f"batch {args.batch} per GPU"
    prec = "fp32" if getattr(args, "dtype", "f32") == "f32" else "bf16 activation storage + bf16 FPN tensor-core operands, fp32 accumulate"
    return f"CISTGCN embed={E} {what}, {shape}, {bs}, {prec}, random-init weights"


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU implementation of the path on the host cores.
    Rank 0 alone works; other ranks exit 0."""
    if rank != 0:
        return
    import torch
    from cistgcn_b200.synth import synth_inputs
    E, V = args.embed, args.joints
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    fn, kind, what = _cpu_forward_fn(E, V, args.mode)
    step_seqs, sub = (1024, 256) if args.mode != "train" else (256, 128)   # bounded sample per step; train batch 128 (train_h36m.yaml:91)
    x, tgt = synth_inputs(step_seqs, V)
    def step():
        for i in range(0, step_seqs, sub):
            fn(x[i:i + sub], tgt[i:i + sub])
    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = time.perf_counter() - t0
    val = step_seqs * args.steps / dt
    sample = f"{args.steps} steps x {step_seqs} sequences (batches of {sub}), E={E}, V={V}, fp32 eval, {args.mode}; {what}; {cores} threads"
    print(json.dumps({
        "impl": "reference", "metric": metric_name(V, args.mode), "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": args.scaling,
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(args, world) + f"; CPU sample of {step_seqs} sequences per step"},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }), flush=True)


def run_native(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    from cistgcn_b200 import _cabi
    from cistgcn_b200.dist import shard_bounds
    from cistgcn_b200.synth import synth_inputs

    E, V = args.embed, args.joints
    mode = args.mode
    # library chatter on stdout (e.g. the "NCCL version" banner) goes to stderr: stdout carries the ONE JSON line
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = _cabi.lib()                                   # fails loudly if the extension is missing
    model = _make_model(E, V).to(dev)
    model.kernel_flags = int(os.environ.get("CISTGCN_BENCH_FLAGS", "0"))
    if args.dtype == "bf16":
        model.act_dtype = torch.bfloat16
    # weak: every rank owns its own --batch sequences; strong: --batch is the global batch, sharded by rank
    if args.scaling == "strong":
        lo, hi = shard_bounds(args.batch, rank, world)
        B, global_B = hi - lo, args.batch
    else:
        B, global_B = args.batch, args.batch * world
    x_host, t_host = synth_inputs(B, V, seed=123 + rank)
    x_pin = x_host.pin_memory()
    pred_pin = torch.empty(B, 25, V, 3).pin_memory()
    x = x_pin.to(dev)
    tgt = t_host.to(dev) if mode == "mpjpe" else None
    tgt_pin = t_host.pin_memory() if mode == "mpjpe" else None
    in_bytes = x.numel() * 4 + (tgt.numel() * 4 if tgt is not None else 0)
    out_bytes = pred_pin.numel() * 4 if mode == "forward" else 25 * 8 + 4

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    count = torch.tensor([float(B * V)], device=dev, dtype=torch.float64)

    def step(xd, td):
        """One pass of the path on device-resident inputs.  mpjpe mode returns (mpjpe_all, mpjpe_per_frame) GLOBAL over
        ranks: per-frame sums (25 doubles) + count all-reduced over NCCL, the only inter-GPU exchange."""
        if mode == "forward":
            return model(xd)[0]
        _, sums = model.forward_mpjpe(xd, td)
        buf = torch.cat([sums, count])
        if world > 1:
            dist.all_reduce(buf, op=dist.ReduceOp.SUM)
        per_frame = buf[:-1] / buf[-1]                         # losses.mpjpe(..., reduce_axis=(0, 2))
        return per_frame.mean(), per_frame                     # reduce_axis=[] and (0, 2)

    # ---- device-resident arm: inputs already in HBM (inputs + activations per step exceed the 126 MB L2 at the
    # benchmark batches; small batches are L2-flushed between steps)
    flush = torch.empty(192 * 1024 * 1024, dtype=torch.uint8, device=dev) if B * 10 * V * 3 * 4 < 160e6 else None
    l2_policy = "inputs_larger_than_L2" if flush is None else "L2 flushed between steps (192 MB memset, outside the events)"
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    for _ in range(max(args.warmup, 3)):
        step(x, tgt)
    barrier()
    sampler.mark()
    lib.cistgcn_profile_enable(1)
    if flush is None:
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        ev0.record()
        for _ in range(args.steps):
            out = step(x, tgt)
        ev1.record()
        barrier()
        ms_local = ev0.elapsed_time(ev1)
    else:
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
        barrier()
        for e0, e1 in evs:
            flush.zero_()
            e0.record()
            out = step(x, tgt)
            e1.record()
        barrier()
        ms_local = sum(e0.elapsed_time(e1) for e0, e1 in evs)
    ms = max_over_ranks(ms_local)
    dump = None
    if args.dump_outputs and rank == 0:                 # before the end-to-end arm runs more steps
        dump = {"pred": _host(_row_sample(out))} if mode == "forward" else \
               {"mpjpe_all": _host(out[0]), "mpjpe_per_frame": _host(out[1])}
    NK = _cabi.PROFILE_KINDS
    kms = (ctypes.c_double * NK)()
    kln = (ctypes.c_int64 * NK)()
    lib.cistgcn_profile_read(kms, kln)
    lib.cistgcn_profile_enable(0)
    clocks = sampler.stop() if rank == 0 else None
    value = global_B * args.steps / (ms / 1e3)
    result_note = None
    if mode == "mpjpe":
        result_note = {"mpjpe_all": float(out[0]), "mpjpe_frame0": float(out[1][0]), "mpjpe_frame24": float(out[1][-1])}

    # ---- end-to-end arm: host buffers; every step copies its inputs host->device and its result device->host inside
    # the timed region.  The step is split into sub-batches so the copies (second stream) overlap the forward of the
    # neighbouring sub-batch -- plain stream pipelining around the public forward().
    # Sub-batches of the kernels' own chunk size (32 768) keep the persistent grids full; the device buffers are double
    # buffered across steps and the two copy directions have their own streams, so a step's H2D runs under the previous
    # step's forward and its D2H under the next one's (every copy is enqueued inside the timed loop; the loop ends when the
    # last D2H has landed).
    n_sub = max(1, B // 32768) if B % 32768 == 0 else (4 if B % 4 == 0 and B >= 4096 else 1)
    sub = B // n_sub
    h2d_stream = torch.cuda.Stream(device=dev)
    d2h_stream = torch.cuda.Stream(device=dev)
    compute_stream = torch.cuda.current_stream(dev)
    x_dev = [[torch.empty(sub, 10, V, 3, device=dev) for _ in range(n_sub)] for _ in range(2)]
    t_dev = [[torch.empty(sub, 25, V, 3, device=dev) for _ in range(n_sub)] for _ in range(2)] if mode == "mpjpe" else None
    res_pin = torch.empty(26, dtype=torch.float64).pin_memory()
    ev_free = [torch.cuda.Event(), torch.cuda.Event()]       # compute no longer reads buffer set p
    for e in ev_free:
        e.record(compute_stream)
    e2e_k = [0]

    def e2e_step():
        par = e2e_k[0] & 1
        e2e_k[0] += 1
        ev_in = [torch.cuda.Event() for _ in range(n_sub)]
        h2d_stream.wait_event(ev_free[par])                  # the step before last is done with this buffer set
        with torch.cuda.stream(h2d_stream):
            for i in range(n_sub):
                x_dev[par][i].copy_(x_pin[i * sub:(i + 1) * sub], non_blocking=True)
                if mode == "mpjpe":
                    t_dev[par][i].copy_(tgt_pin[i * sub:(i + 1) * sub], non_blocking=True)
                ev_in[i].record(h2d_stream)
        if mode == "forward":
            for i in range(n_sub):
                compute_stream.wait_event(ev_in[i])
                pr = model(x_dev[par][i])[0]
                ev_out = torch.cuda.Event()
                ev_out.record(compute_stream)
                pr.record_stream(d2h_stream)
                with torch.cuda.stream(d2h_stream):
                    d2h_stream.wait_event(ev_out)
                    pred_pin[i * sub:(i + 1) * sub].copy_(pr, non_blocking=True)
        else:
            tot = torch.zeros(26, device=dev, dtype=torch.float64)
            for i in range(n_sub):
                compute_stream.wait_event(ev_in[i])
                _, sums = model.forward_mpjpe(x_dev[par][i], t_dev[par][i])
                tot[:25] += sums
            tot[25] = float(B * V)
            if world > 1:
                dist.all_reduce(tot, op=dist.ReduceOp.SUM)
            res_pin.copy_(tot, non_blocking=True)            # per-frame sums + count: the step's result, read on the host
        ev_free[par].record(compute_stream)

    def e2e_drain():
        compute_stream.wait_stream(d2h_stream)               # the last D2H has landed

    for _ in range(2):
        e2e_step()
    e2e_drain()
    barrier()
    def e2e_timed():
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for _ in range(args.steps):
            e2e_step()
        e2e_drain()
        ev1.record()
        barrier()
        return max_over_ranks(ev0.elapsed_time(ev1))

    ms_e2e = e2e_timed()
    if ms_e2e < 200.0:          # a K-step region this short (small batches) is at the mercy of one host hiccup: median of 5
        ms_e2e = sorted([ms_e2e] + [e2e_timed() for _ in range(4)])[2]
    e2e_value = global_B * args.steps / (ms_e2e / 1e3)
    if mode == "forward":
        checksum = float(pred_pin[:16].double().abs().sum())          # the D2H result is really read
    else:
        checksum = float((res_pin[:25] / res_pin[25]).mean())

    if world > 1:
        dist.destroy_process_group()
    if rank != 0:
        return

    hbm_peak, peak_src = measured_peaks()
    names = [lib.cistgcn_profile_kind_name(i).decode() for i in range(NK)]
    launches = sum(int(v) for v in kln)                     # launches of OUR kernels inside the timed region
    fpn_tc = V in (22, 18) and not (model.kernel_flags & _cabi.FLAG_FPN_FP32)
    kshare = {names[i]: {"ms_per_step": kms[i] / args.steps, "launches_per_step": int(kln[i]) / args.steps}
              for i in range(NK) if kln[i]}
    if "fpn_kernel" in kshare:
        kshare["fpn_kernel"]["variant"] = "fpn_tc_kernel (tcgen05)" if fpn_tc else "fpn_chain_kernel (FP32 FMA)"
    dom = max(range(NK), key=lambda i: kms[i])
    total_kms = sum(kms)
    n_launch_dom = max(int(kln[dom]), 1)
    seqs = B * args.steps                                   # sequences pushed through every kernel kind on this rank
    kb = stage_bytes_per_seq(E, V, act_bytes=2 if args.dtype == "bf16" else 4)
    fl_total = FLOPS_PER_SEQ.get((V, E), 0.0)
    dstd_flops = fl_total - FPN_FLOPS_PER_SEQ[V] - 0.7e6 * V / 22
    dur_s = kms[dom] / 1e3 / n_launch_dom                   # average launch duration, CUDA events on the launch stream
    bytes_launch = kb.get(names[dom], 0) * seqs / n_launch_dom
    achieved = bytes_launch / dur_s / 1e9
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "dram_traffic.json")
    if os.path.isfile(tpath):                               # ncu --set full capture of the same launch shape, bytes / sequence
        tj = json.load(open(tpath)).get(f"E{E}_V{V}", {}).get(names[dom])
        if tj is not None:
            traffic = tj * seqs / n_launch_dom
    roofline = {"bound": "hbm", "kernel": names[dom], "achieved": achieved, "peak": hbm_peak, "unit": "GB/s",
                "frac": achieved / hbm_peak, "traffic": traffic, "peak_source": peak_src,
                "share_of_step": kms[dom] / total_kms if total_kms else None,
                "bytes_per_launch": bytes_launch, "launch_ms": dur_s * 1e3,
                "note": "the fp32 path is bound by the FP32 FMA pipe, not HBM (SURVEY.md 0.3 / 8d): see roofline_fp32_fma"}
    # FP32-FMA view: all DSTD kinds together (their FLOPs cannot be split per stage from the reference's counter)
    dstd_ms = sum(kms[i] for i in range(NK) if names[i].startswith("dstd_"))
    dstd_tf = dstd_flops * seqs / (dstd_ms / 1e3) / 1e12 if dstd_ms else 0.0
    roofline_fma = {"bound": "fp32_fma", "kernel": "dstd_* (all DSTD-GC stages)", "achieved": dstd_tf, "peak": FP32_FMA_PEAK_TFLOPS,
                    "unit": "TFLOP/s", "frac": dstd_tf / FP32_FMA_PEAK_TFLOPS,
                    "share_of_step": dstd_ms / total_kms if total_kms else None,
                    "peak_source": "nominal 148 SM x 128 lanes x 2 x 1.965 GHz; measured ceiling of a pure FFMA loop on this "
                                   "pool is 92/128 of it (profiles/microbench_r1.log)",
                    "whole_forward": {"achieved": fl_total * (value / world) / 1e12,
                                      "frac": fl_total * (value / world) / 1e12 / FP32_FMA_PEAK_TFLOPS,
                                      "hbm_frac_survey_bytes": bytes_per_seq(V, E) * (value / world) / 1e9 / hbm_peak}}
    roofline_tensor = None
    if fpn_tc and kln[1]:
        tpeak, tsrc = measured_tensor_peak()
        fpn_s = kms[1] / 1e3
        alg = FPN_FLOPS_PER_SEQ[V] * seqs / fpn_s / 1e12
        issued = fpn_tc_issued_flops_per_seq() * seqs / fpn_s / 1e12
        roofline_tensor = {"bound": "tensor", "kernel": "fpn_tc_kernel", "achieved": alg, "issued": issued, "peak": tpeak,
                           "unit": "TFLOP/s", "frac": alg / tpeak, "frac_issued": issued / tpeak, "peak_source": tsrc,
                           "share_of_step": kms[1] / total_kms if total_kms else None,
                           "launch_ms": kms[1] / max(int(kln[1]), 1),
                           "note": "achieved = the reference's algorithmic FPN FLOPs (SURVEY.md 8d) / kernel time; issued = tcgen05 "
                                   "FLOPs incl. channel padding to 32 and the split-operand products that buy fp32 accuracy "
                                   "(x1*[w1|w2|w3] + x2*wh); the pipe is fed from shared memory at N <= 96, see DESIGN.md"}
    line = {
        "metric": metric_name(V, mode), "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": args.scaling,
        "vs_baseline": None, "dtype": args.dtype, "data": "synthetic",
        "config": {"workload": workload_name(args, world), "batch_per_gpu": B, "global_batch": global_B, "embed": E,
                   "joints": V, "mode": mode,
                   "parallelism": f"batch-sharded x{world}, no data-path collective" +
                                  ("; MPJPE frame sums: one 208-byte NCCL all-reduce per step" if mode == "mpjpe" and world > 1 else ""),
                   "l2_policy": l2_policy, "kernel_flags": model.kernel_flags},
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": in_bytes, "d2h_bytes_per_step": out_bytes,
                "ms_per_step": ms_e2e / args.steps,
                "api": f"CISTGCN.{'forward' if mode == 'forward' else 'forward_mpjpe'} on pinned host buffers, {n_sub} sub-batches, H2D / D2H on their own streams, device buffers double-buffered across steps",
                "checksum": checksum},
        "gpu_launches": launches * world,     # every rank launches the same kernels on its own GPU
        "kernels": kshare,
        "roofline": roofline,
        "roofline_fp32_fma": roofline_fma,
        "roofline_tensor": roofline_tensor,
        "clocks": clocks,
    }
    if result_note:
        line["result"] = result_note
    if world == 1:
        line["cpu_baseline"] = cpu_baseline(E, V, mode, args.cpu_budget)
    if dump is not None:
        write_dump(args.dump_outputs, dump)
    sys.stdout.flush()
    os.dup2(saved_stdout, 1)
    print(json.dumps(line), flush=True)


def run_train(args, rank, world, local_rank):
    """configs[4]: the reference's training step (environment/train.py:54-107) data-parallel over the ranks: train-mode
    forward with local batch-statistics BatchNorm (the reference has no SyncBN), losses.mpjpe (reduce_axis=[]), backward,
    ONE NCCL all-reduce of the flat fp32 gradient buffer, fused Adam (lr .01, weight decay 1e-4 in the gradient)."""
    import torch
    import torch.distributed as dist
    from cistgcn_b200 import CISTGCN, _cabi
    from cistgcn_b200.synth import make_opt, synth_inputs
    from cistgcn_b200.train import Trainer

    E, V, B = args.embed, args.joints, args.batch
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    opt = make_opt(E, V, dropout=0.1)                        # learning_config.dropout of train_h36m.yaml
    torch.manual_seed(0)
    model = CISTGCN(opt.architecture_config, opt.learning_config).to(dev).train()
    tr = Trainer(model, lr=0.01, weight_decay=1e-4, cuda_graph=not args.no_graph)
    tr.graph.seed += rank                                    # every replica draws its own dropout masks
    x_host, t_host = synth_inputs(B, V, seed=123 + rank)
    x_pin, t_pin = x_host.pin_memory(), t_host.pin_memory()
    x, tgt = x_pin.to(dev), t_pin.to(dev)
    res_pin = torch.empty(25, dtype=torch.float64).pin_memory()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    flush = torch.empty(192 * 1024 * 1024, dtype=torch.uint8, device=dev)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    for _ in range(max(args.warmup, 3)):                     # (with --graph: step 1 eager, step 2 captures, step 3.. replay)
        tr.step(x, tgt)
    barrier()
    sampler.mark()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    ar = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    for (e0, e1), (a0, a1) in zip(evs, ar):
        flush.zero_()
        e0.record()
        sums = tr.step(x, tgt, timing=(a0, a1))
        e1.record()
    barrier()
    ms = max_over_ranks(sum(e0.elapsed_time(e1) for e0, e1 in evs))
    ar_ms = max_over_ranks(sum(a0.elapsed_time(a1) for a0, a1 in ar)) if world > 1 else 0.0
    dump = None
    if args.dump_outputs and rank == 0:                 # before the end-to-end arm runs more steps
        dump = {"frame_sums": _host(sums), "parameters": _host(tr.flat.flat)}
    launches = tr.graph.launches + 1 + (1 if world > 1 else 0)
    clocks = sampler.stop() if rank == 0 else None
    value = world * B * args.steps / (ms / 1e3)
    loss = float(sums.sum() / (B * 25 * V))

    # end to end: inputs and targets from pinned host memory every step, the loss read back on the host
    def e2e_step():
        x.copy_(x_pin, non_blocking=True)
        tgt.copy_(t_pin, non_blocking=True)
        s = tr.step(x, tgt)
        res_pin.copy_(s, non_blocking=True)
    for _ in range(2):
        e2e_step()
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(args.steps):
        e2e_step()
    ev1.record()
    barrier()
    ms_e2e = max_over_ranks(ev0.elapsed_time(ev1))
    e2e_value = world * B * args.steps / (ms_e2e / 1e3)
    if world > 1:
        dist.destroy_process_group()
    if rank != 0:
        return
    n_params = tr.flat.numel
    line = {
        "metric": metric_name(V, "train"), "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(args, world), "batch_per_gpu": B, "global_batch": B * world, "embed": E, "joints": V,
                   "mode": "train", "dropout": 0.1, "optimizer": "Adam lr 0.01 wd 1e-4 (environment/utils.py:53-57)",
                   "parallelism": f"data-parallel x{world}, local BatchNorm statistics, one all-reduce of {4 * n_params} bytes per step",
                   "l2_policy": "L2 flushed between steps (192 MB memset, outside the events)",
                   "cuda_graph": bool(tr.use_cuda_graph)},
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": (x.numel() + tgt.numel()) * 4, "d2h_bytes_per_step": 25 * 8,
                "ms_per_step": ms_e2e / args.steps, "api": "Trainer.step on pinned host inputs + loss read-back", "checksum": float(res_pin.sum())},
        "gpu_launches": launches * world * args.steps,
        "launches_per_step": launches,
        "collective": {"kind": "ncclAllReduce(SUM) over the flat fp32 gradient buffer" if world > 1 else "none (1 rank)",
                       "bytes": 4 * n_params, "ms_per_step": ar_ms / args.steps, "share_of_step": (ar_ms / ms) if ms else None},
        "result": {"loss_last_step": loss},
        "roofline": {"bound": "hbm", "kernel": "training step (about 2 600 layer kernels per step)", "achieved": None, "peak": measured_peaks()[0],
                     "unit": "GB/s", "frac": None, "traffic": None,
                     "note": "launch-bound: whole-batch BatchNorm statistics force layer-by-layer kernels; see DESIGN.md"},
        "clocks": clocks,
    }
    if world == 1:
        line["cpu_baseline"] = cpu_baseline(E, V, "train", args.cpu_budget, batch=B)
    if dump is not None:
        write_dump(args.dump_outputs, dump)
    sys.stdout.flush()
    os.dup2(saved_stdout, 1)
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--embed", type=int, default=32)
    ap.add_argument("--joints", type=int, default=22)
    ap.add_argument("--batch", type=int, default=65536, help="sequences per GPU per step (weak) / global batch (strong)")
    ap.add_argument("--mode", default="forward", choices=["forward", "mpjpe", "train"])
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--dtype", default="f32", choices=["f32", "bf16"],
                    help="bf16: cistgcn_forward_bf16 (bf16 activation storage + single-term bf16 FPN tensor-core operands)")
    ap.add_argument("--no-graph", action="store_true", help="train mode: launch every layer kernel from the host instead of "
                    "replaying the captured CUDA graph of forward + loss + backward")
    ap.add_argument("--cpu-budget", type=float, default=12.0, help="seconds of CPU baseline timing (N=1 only)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's results to DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the native path's results; it does not apply to --impl reference")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    if args.gpus > 1 and world == 1:
        # convenience: re-launch under torchrun
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", "29517", os.path.abspath(__file__)] + sys.argv[1:]
        raise SystemExit(subprocess.call(cmd))
    if args.impl == "reference":
        run_reference(args, rank, world)
    elif args.mode == "train":
        run_train(args, rank, world, local_rank)
    else:
        run_native(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
