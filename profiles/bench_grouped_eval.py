"""Cost of grouped evaluation (per-group per-frame tables in one pass, csrc/eval_grouped.cu).

usage: python profiles/bench_grouped_eval.py [--steps K] [--warmup W] [--rounds R] [--out FILE]

Runs (E = 32, 22 joints, total batch 65 536 split over G = 15 groups; device-resident inputs, x and the target both
larger than the 126 MB L2; CUDA events around K steps, arms of a run alternate, R rounds in this process):
  forward_f32 / forward_bf16   output_n = 25:
      ungrouped        forward_mpjpe(x, t)                       (fused MPJPE in the tail kernel)
      grouped          forward_mpjpe(x, t, groups, 15)           (forward + one grouped_mpjpe_kernel pass)
      per_group_loop   15 x forward_mpjpe(x_g, t_g) on the test set split by group beforehand
  rollout_metrics_f32          long-term model (output_n = 25) rolled out to 50 frames:
      rollout          rollout(x, 50)
      rollout_metrics  rollout(x, 50) + EvalMetrics(50, n_groups=15).compute(out, t, groups=groups)
Before timing, the grouped sums are compared with the per-group loop at the timed size (max relative difference in
the JSON).  A second, profiled pass per arm gives per-kernel-kind milliseconds (cistgcn_profile_read; grouped_mpjpe_kernel
counts under "mpjpe_kernel").  One JSON line per measurement on stdout (and appended to --out); the first line names the
card and its power limit."""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from cistgcn_b200 import CISTGCN, _cabi  # noqa: E402
from cistgcn_b200.metrics import EvalMetrics, source_map  # noqa: E402
from cistgcn_b200.synth import make_opt, synth_inputs  # noqa: E402

DEV = torch.device("cuda", 0)
E, V, B, G = 32, 22, 65536, 15
H_ROLL = 50


def emit(rec, out):
    line = json.dumps(rec)
    print(line, flush=True)
    if out:
        with open(out, "a") as f:
            f.write(line + "\n")


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(DEV), "nvidia_smi": q.stdout.strip() or q.stderr.strip()}


def model_for(To, dtype):
    opt = make_opt(E, V, output_n=To)
    torch.manual_seed(0)
    m = CISTGCN(opt.architecture_config, opt.learning_config).eval().to(DEV)
    if dtype == "bf16":
        m.act_dtype = torch.bfloat16
    return m


def profile(lib, fn, reps=2):
    NK = _cabi.PROFILE_KINDS
    names = [lib.cistgcn_profile_kind_name(k).decode() for k in range(NK)]
    torch.cuda.synchronize(DEV)
    lib.cistgcn_profile_enable(1)
    for _ in range(reps):
        fn()
    kms, kln = (ctypes.c_double * NK)(), (ctypes.c_int64 * NK)()
    _cabi.check(lib.cistgcn_profile_read(kms, kln), "profile_read", lib)
    lib.cistgcn_profile_enable(0)
    return {names[k]: round(kms[k] / reps, 4) for k in range(NK) if kln[k]}


def time_arms(steps, args):
    for fn in steps.values():
        for _ in range(args.warmup):
            fn()
    times = {arm: [] for arm in steps}
    for _ in range(args.rounds):
        for arm, fn in steps.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize(DEV)
            e0.record()
            for _ in range(args.steps):
                fn()
            e1.record()
            torch.cuda.synchronize(DEV)
            times[arm].append(e0.elapsed_time(e1) / args.steps)
    return times


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    lib = _cabi.lib()
    emit({"card": card()}, args.out)
    groups = torch.randint(0, G, (B,), generator=torch.Generator().manual_seed(0)).to(DEV)
    with torch.no_grad():
        for dtype in ("f32", "bf16"):
            m = model_for(25, dtype)
            x, t = synth_inputs(B, V, output_n=25)
            x, t = x.to(DEV), t.to(DEV)
            xs = [x[groups == g].contiguous() for g in range(G)]
            ts = [t[groups == g].contiguous() for g in range(G)]
            _, sums, counts = m.forward_mpjpe(x, t, groups, G)
            loop = torch.stack([m.forward_mpjpe(xg, tg)[1] for xg, tg in zip(xs, ts)])
            rel = float(((sums - loop).abs() / loop.abs()).max())

            def per_group_loop():
                return [m.forward_mpjpe(xg, tg) for xg, tg in zip(xs, ts)]

            steps = {"ungrouped": lambda: m.forward_mpjpe(x, t), "grouped": lambda: m.forward_mpjpe(x, t, groups, G),
                     "per_group_loop": per_group_loop}
            times = time_arms(steps, args)
            base = statistics.median(times["ungrouped"])
            for arm in steps:
                ms = statistics.median(times[arm])
                emit({"run": f"forward_{dtype}", "arm": arm, "embed": E, "joints": V, "output_n": 25, "batch": B,
                      "groups": G, "dtype": dtype, "seq_per_s": round(B / (ms / 1e3)), "ms_per_step": round(ms, 4),
                      "ms_per_step_rounds": [round(v, 4) for v in times[arm]],
                      "ratio_to_ungrouped": round(ms / base, 4), "grouped_vs_loop_max_rel_diff": rel,
                      "kernel_ms": profile(lib, steps[arm])}, args.out)
            del steps, m, x, t, xs, ts
            torch.cuda.empty_cache()

        m = model_for(25, "f32")
        x, t = synth_inputs(B, V, output_n=H_ROLL)
        x, t = x.to(DEV), t.to(DEV)
        smap = source_map(V, list(range(V)))
        bones = [(j, j + 1) for j in range(V - 1)]
        ev = EvalMetrics(H_ROLL, smap, bones, n_groups=G)

        def rollout_metrics():
            ev.compute(m.rollout(x, H_ROLL), t, groups=groups)

        steps = {"rollout": lambda: m.rollout(x, H_ROLL), "rollout_metrics": rollout_metrics}
        times = time_arms(steps, args)
        base = statistics.median(times["rollout"])
        for arm in steps:
            ms = statistics.median(times[arm])
            emit({"run": "rollout_metrics_f32", "arm": arm, "embed": E, "joints": V, "output_n": 25, "horizon": H_ROLL,
                  "batch": B, "groups": G, "dtype": "f32", "seq_per_s": round(B / (ms / 1e3)), "ms_per_step": round(ms, 4),
                  "ms_per_step_rounds": [round(v, 4) for v in times[arm]], "ratio_to_rollout": round(ms / base, 4),
                  "kernel_ms": profile(lib, steps[arm])}, args.out)
        vals = ev.values_by_group()
        emit({"run": "rollout_metrics_f32", "check": "values_by_group finite",
              "ok": all(bool(torch.isfinite(v).all()) for v in vals.values())}, args.out)


if __name__ == "__main__":
    main()
