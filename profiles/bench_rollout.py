"""Sequences/s of a 25-frame (1 s at 25 fps) forecast three ways: a short-term model (output_n = 10) rolled out on the
device (CISTGCN.rollout), a long-term model (output_n = 25) in one forward, and the same rollout as a Python loop over
the short-term model's forward.

usage: python profiles/bench_rollout.py [--steps K] [--warmup W] [--rounds R] [--out FILE]

Runs (device-resident inputs, every input tensor larger than the 126 MB L2; CUDA events around K steps):
  e32_v22_f32     E = 32, 22 joints, batch 65 536, fp32
  e32_v22_bf16    same, act_dtype = bfloat16 (cistgcn_rollout_bf16 / cistgcn_forward_bf16)
  mpjpe_e64_v18   E = 64, 18 joints, batch 262 144, with MPJPE over the 25 frames: rollout_mpjpe / forward_mpjpe /
                  the loop followed by losses.mpjpe(reduce_axis=(0, 2))
Arms of a run alternate, R rounds in this process.  Before timing, the device rollout is checked bit for bit against the
Python loop.  A second, profiled pass per arm gives per-kernel-kind milliseconds (cistgcn_profile_read); the rollout's
frame-moving kernel is the "other" kind.  One JSON line per measurement on stdout (and appended to --out); the first
line names the card and its power limit."""
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
from cistgcn_b200.losses import mpjpe  # noqa: E402
from cistgcn_b200.synth import make_opt, synth_inputs  # noqa: E402

DEV = torch.device("cuda", 0)
H = 25
RUNS = [("e32_v22_f32", 32, 22, 65536, "forward", "f32"),
        ("e32_v22_bf16", 32, 22, 65536, "forward", "bf16"),
        ("mpjpe_e64_v18", 64, 18, 262144, "mpjpe", "f32")]
ARMS = ("rollout_10", "forward_25", "loop_10")


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


def model_for(E, V, To, dtype):
    opt = make_opt(E, V, output_n=To)
    torch.manual_seed(0)
    m = CISTGCN(opt.architecture_config, opt.learning_config).eval().to(DEV)
    if dtype == "bf16":
        m.act_dtype = torch.bfloat16
    return m


def python_loop(m, x):
    """The rollout as a user writes it around forward: the last input_n frames of cat(window, prediction) feed the next
    step; the predictions are concatenated and cut to the horizon."""
    w, preds = x, []
    for _ in range(-(-H // m.n_output)):
        p = m(w)[0]
        preds.append(p)
        w = torch.cat([w, p], 1)[:, -m.n_input:]
    return torch.cat(preds, 1)[:, :H]


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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    lib = _cabi.lib()
    emit({"card": card()}, args.out)
    with torch.no_grad():
        for name, E, V, B, mode, dtype in RUNS:
            m10, m25 = model_for(E, V, 10, dtype), model_for(E, V, 25, dtype)
            x, t = synth_inputs(B, V, output_n=H)
            x, t = x.to(DEV), t.to(DEV)
            if mode == "forward":
                steps = {"rollout_10": lambda: m10.rollout(x, H), "forward_25": lambda: m25(x),
                         "loop_10": lambda: python_loop(m10, x)}
            else:
                def loop_mpjpe():
                    p = python_loop(m10, x)
                    return p, mpjpe(p, t, reduce_axis=(0, 2))
                steps = {"rollout_10": lambda: m10.rollout_mpjpe(x, t), "forward_25": lambda: m25.forward_mpjpe(x, t),
                         "loop_10": loop_mpjpe}
            bitwise = torch.equal(m10.rollout(x, H), python_loop(m10, x))
            for arm in ARMS:
                for _ in range(args.warmup):
                    steps[arm]()
            times = {arm: [] for arm in ARMS}
            for _ in range(args.rounds):
                for arm in ARMS:
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    torch.cuda.synchronize(DEV)
                    e0.record()
                    for _ in range(args.steps):
                        steps[arm]()
                    e1.record()
                    torch.cuda.synchronize(DEV)
                    times[arm].append(e0.elapsed_time(e1) / args.steps)
            for arm in ARMS:
                ms = statistics.median(times[arm])
                emit({"run": name, "arm": arm, "horizon": H, "embed": E, "joints": V, "batch": B, "mode": mode,
                      "dtype": dtype, "seq_per_s": round(B / (ms / 1e3)), "ms_per_step": round(ms, 4),
                      "ms_per_step_rounds": [round(v, 4) for v in times[arm]],
                      "rollout_bitwise_equals_loop": bitwise, "kernel_ms": profile(lib, steps[arm])}, args.out)
            del steps, m10, m25, x, t
            torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
