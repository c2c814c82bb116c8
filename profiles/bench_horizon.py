"""Sequences/s of the inference path at the two supported horizons, output_n = 10 (short term) and 25 (long term).

usage: python profiles/bench_horizon.py [--steps K] [--warmup W] [--rounds R] [--out FILE]

Runs (device-resident inputs, every input tensor larger than the 126 MB L2; CUDA events around K steps):
  fwd_e32_v22_f32   E = 32, 22 joints, batch 65 536, forward, fp32
  fwd_e32_v22_bf16  same, cistgcn_forward_bf16
  mpjpe_e64_v18     E = 64, 18 joints, batch 262 144, forward + fused MPJPE (bench.py --mode mpjpe)
Each run is timed at output_n = 10 and 25 in turn, R rounds alternating in this process.  A second, profiled pass per
run gives per-kernel-kind milliseconds (cistgcn_profile_read).  Then stage 3 of the output block alone
(cistgcn_dstd_block_f32): the warp-per-sample kernel (default flags) against the tile kernel (CISTGCN_FLAG_DSTD_MIX_FFMA).
One JSON line per measurement on stdout (and appended to --out); the first line names the card and its power limit."""
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
from cistgcn_b200.synth import make_opt, synth_inputs  # noqa: E402

DEV = torch.device("cuda", 0)
RUNS = [("fwd_e32_v22_f32", 32, 22, 65536, "forward", "f32"),
        ("fwd_e32_v22_bf16", 32, 22, 65536, "forward", "bf16"),
        ("mpjpe_e64_v18", 64, 18, 262144, "mpjpe", "f32")]


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


def profile(lib, fn, reps=3):
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
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    lib = _cabi.lib()
    emit({"card": card()}, args.out)
    with torch.no_grad():
        for name, E, V, B, mode, dtype in RUNS:
            arms = {}
            for To in (10, 25):
                m = model_for(E, V, To, dtype)
                x, t = synth_inputs(B, V, output_n=To)
                x, t = x.to(DEV), t.to(DEV)
                step = (lambda m=m, x=x: m(x)) if mode == "forward" else (lambda m=m, x=x, t=t: m.forward_mpjpe(x, t))
                for _ in range(args.warmup):
                    step()
                arms[To] = (m, step, [])
            for _ in range(args.rounds):
                for To in (10, 25):
                    _, step, times = arms[To]
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    torch.cuda.synchronize(DEV)
                    e0.record()
                    for _ in range(args.steps):
                        step()
                    e1.record()
                    torch.cuda.synchronize(DEV)
                    times.append(e0.elapsed_time(e1) / args.steps)
            for To in (10, 25):
                m, step, times = arms[To]
                ms = statistics.median(times)
                emit({"run": name, "output_n": To, "embed": E, "joints": V, "batch": B, "mode": mode, "dtype": dtype,
                      "seq_per_s": round(B / (ms / 1e3)), "ms_per_step": round(ms, 4),
                      "ms_per_step_rounds": [round(v, 4) for v in times], "fpn_tc": m.pack().fpn_tc,
                      "kernel_ms": profile(lib, step)}, args.out)
            del arms
            torch.cuda.empty_cache()
        # stage 3 of the output block on its own: warp-per-sample (default) vs tile kernel (MIX_FFMA)
        stream = torch.cuda.current_stream(DEV).cuda_stream
        for V, B in ((22, 65536), (18, 262144)):
            for To in (10, 25):
                pk = model_for(8, V, To, "f32").pack()
                d = pk.block_desc("out", 0)
                xin = torch.randn(B, 3 * V * To, device=DEV)
                out = torch.empty_like(xin)
                ws = torch.empty(lib.cistgcn_dstd_block_workspace_bytes(d, B), dtype=torch.uint8, device=DEV)
                rec = {"run": "out_block_stage3", "output_n": To, "joints": V, "batch": B}
                for label, flags in (("default", 0), ("tile", _cabi.FLAG_DSTD_MIX_FFMA)):
                    def run(flags=flags):
                        _cabi.check(lib.cistgcn_dstd_block_f32(d, pk.blob.data_ptr(), xin.data_ptr(), out.data_ptr(), B, None,
                                                               ws.data_ptr(), ws.numel(), flags, stream), "dstd_block", lib)
                    for _ in range(args.warmup):
                        run()
                    rec[label] = [profile(lib, run, reps=args.steps) for _ in range(args.rounds)]
                emit(rec, args.out)


if __name__ == "__main__":
    main()
