#!/usr/bin/env python
"""Time one environment step of the policy: `PolicyActor.step` (one graph replay) against the eager L = 1 loop.

    python tools/bench_act.py [--steps 2000] [--warmup 50] [--rounds 4] [--out FILE]

Per case (encoder x n_envs, the benchmark's policy arguments: width 256, S = 9, A = 6, SAC) three arms, alternated in
`--rounds` blocks of steps/rounds steps each, host wall time per step including the H2D copy of the inputs, the D2H copy
of the outputs and the wait:
  eager_parent : policy.forward at L = 1 under no_grad with the state carried, decode kernels off (the path before
                 rorl_small_linear and the fused Mamba step: tensor-core GEMM / cuBLAS / the torch Mamba step chain);
  eager        : the same loop with the decode kernels on;
  actor        : alg.make_actor(n_envs).step(...).
`launches` is the number of this library's kernels per step (`_native.launch_count()`; torch's own kernels are not
counted).  Also `rorl_small_linear` alone at the in_proj shape [n_envs, 256] x [1024, 256]^T, CUDA events around 2000 eager
back-to-back calls through the Python wrapper (so the figure is bounded below by the host's enqueue rate), next to the
tensor-core GEMM (passes 2, with its pre-split) called the same way.  The card's name and power limit are recorded in the first line.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

ENCODERS = ["smamba_s32_c16_b2_nln", "gilr", "gru", "lstm"]
N_ENVS = [1, 16, 64]


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
    except Exception as e:                                                   # noqa: BLE001
        q = f"nvidia-smi unavailable: {e}"
    import torch
    return {"card": torch.cuda.get_device_name(0), "nvidia_smi": q}


def build_engine(enc, dev):
    import torch
    from bench import HP, model_kwargs
    from rorl_b200.algorithm.sac_full_length_rnn_redq_sep_optim import SACFullLengthRNNREDQ_SEP_OPTIM
    torch.manual_seed(0)
    np.random.seed(0)
    return SACFullLengthRNNREDQ_SEP_OPTIM(dict(HP), model_kwargs(enc, False), model_kwargs(enc, True), 1000, device=dev)


def time_case(alg, n, steps, warmup, rounds, dev):
    import torch
    import rorl_b200._native as NV
    import rorl_b200.kernels as K
    S, A = alg.policy.state_dim, alg.policy.action_dim
    gen = np.random.default_rng(0)
    inputs = [(gen.standard_normal((n, S)).astype(np.float32), gen.standard_normal((n, S)).astype(np.float32),
               np.tanh(gen.standard_normal((n, A))).astype(np.float32)) for _ in range(64)]
    actor = alg.make_actor(n)
    state = {"h": alg.policy.make_init_state(n, dev)}

    def eager(i):
        st, ls, la = inputs[i % 64]
        t = [torch.from_numpy(v).to(dev, non_blocking=False).view(n, 1, -1) for v in (st, ls, la)]
        with torch.no_grad():
            out = alg.policy.forward(t[0], t[1], t[2], state["h"])
        state["h"] = out[4]
        return out[0].cpu().numpy(), out[2].cpu().numpy(), out[3].cpu().numpy()

    def act(i):
        st, ls, la = inputs[i % 64]
        return actor.step(st, ls, la, None, None)

    arms = {"eager_parent": (eager, False), "eager": (eager, True), "actor": (act, True)}
    times = {k: [] for k in arms}
    launches = {}
    for name, (fn, on) in arms.items():                                      # warm-up (the actor captures here)
        K.DECODE_STEP_KERNELS = on
        for i in range(warmup):
            fn(i)
        torch.cuda.synchronize()
        l0 = NV.launch_count()
        fn(0)
        launches[name] = NV.launch_count() - l0
    per = steps // rounds
    for r in range(rounds):
        for name, (fn, on) in arms.items():
            K.DECODE_STEP_KERNELS = on
            torch.cuda.synchronize()
            for i in range(per):
                t0 = time.perf_counter()
                fn(i)
                times[name].append(time.perf_counter() - t0)
    K.DECODE_STEP_KERNELS = True
    res = {f"{k}_us_median": round(float(np.median(v)) * 1e6, 2) for k, v in times.items()}
    res.update({f"{k}_us_p90": round(float(np.percentile(v, 90)) * 1e6, 2) for k, v in times.items()})
    res.update({f"{k}_launches": v for k, v in launches.items()})
    res["steps_per_arm"] = per * rounds
    return res


def time_small_linear(n, dev, iters=2000):
    import torch
    import rorl_b200.kernels as K
    x = torch.randn(n, 256, device=dev)
    W = torch.randn(1024, 256, device=dev)
    out = {}
    for name, fn in (("small_linear", lambda: K.small_linear(x, W)), ("gemm_tn_passes2", lambda: K.gemm_tn(x, W))):
        for _ in range(50):
            fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(iters):
            fn()
        e1.record()
        torch.cuda.synchronize()
        out[f"{name}_us"] = round(e0.elapsed_time(e1) * 1e3 / iters, 3)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=50)
    ap.add_argument("--rounds", type=int, default=4)
    ap.add_argument("--encoders", default=",".join(ENCODERS))
    ap.add_argument("--envs", default=",".join(map(str, N_ENVS)))
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    assert torch.cuda.is_available(), "bench_act.py measures on the GPU"
    dev = torch.device("cuda", 0)
    lines = [dict(kind="card", **card())]
    for n in map(int, args.envs.split(",")):
        lines.append(dict(kind="small_linear", shape=f"[{n}, 256] x [1024, 256]^T", n_envs=n, **time_small_linear(n, dev)))
        print(json.dumps(lines[-1]), flush=True)
    for enc in args.encoders.split(","):
        alg = build_engine(enc, dev)
        for n in map(int, args.envs.split(",")):
            lines.append(dict(kind="act", encoder=enc, n_envs=n, **time_case(alg, n, args.steps, args.warmup, args.rounds, dev)))
            print(json.dumps(lines[-1]), flush=True)
        del alg
        torch.cuda.empty_cache()
    print(json.dumps(lines[0]))
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(json.dumps(l) for l in lines) + "\n")


if __name__ == "__main__":
    main()
