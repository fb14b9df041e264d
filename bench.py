#!/usr/bin/env python
"""Benchmark of the recurrent off-policy update hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

A "step" is one complete SAC update (`train_one_batch`: sample -> target Q -> critic step + Polyak ->
actor step -> alpha step; 5 encoder forwards, 2 backwards) with the smamba_s32_c16_b2_nln encoder on a
synthetic HalfCheetah-V-shaped replay (obs 9, act 6) of 32 full 1000-step trajectories PER GPU
(weak scaling: N GPUs update on 32*N trajectories, trajectory-sharded, NCCL gradient all-reduce).
Metric: trajectory-steps/s = valid transitions updated on per second, whole job.

  value  : K updates with the replay resident in HBM (host plan + device gather inside the step), CUDA events,
           max over ranks.  From the third update on the step is replayed from captured CUDA-graph segments (the
           public API's default; RORL_CUDA_GRAPH=0 keeps the eager launch sequence); `gpu_launches` counts the
           kernels of this library launched or replayed inside the timed region.
  e2e    : same update through the public API fed from HOST memory, the way the reference feeds it: per step a
           pinned host batch is copied H2D and the logged scalars are read back D2H, inside the timed region.
  roofline: the selective-scan kernel (forward or backward, whichever takes the larger share), timed alone
           with CUDA events on its launch stream at the workload's shape.
  cpu_baseline: the reference's OWN `train_one_batch` (unmodified code staged under oracle/_ref by oracle/make_ref.py;
           kind "reference"; the oracle port, kind "port", only if that copy is missing) with the GRU encoder -- the
           reference's CPU-runnable configuration -- on the same 32x1000 shape and on config 1's 8x200 shape, on this
           box's host cores.
  strong_scaling: the BASELINE config-5 job (256 trajectories x 1000 steps GLOBAL, 256/N per GPU) timed the same way.
`--impl reference` times the reference's own CPU implementation of THIS arm's configuration (same encoder, 32 rows,
same widths; on CPU its smamba layer walks `Mamba.step` once per time step) on a bounded sample: every trajectory is
cut to RORL_REF_TLEN (default 100) of its 1000 steps -- the per-step Python loop is linear in the trajectory length,
so steps/s of the sample is steps/s of the workload, while the row count (what the loop amortises over) is the real 32.
`--dump-outputs DIR` writes what the last timed update of the `value` arm computed as .npy files (see `dump_outputs`).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

S_DIM, A_DIM, T_LEN, N_TRAJ = 9, 6, 1000, 32
STRONG_TRAJ = 256
ENCODER = os.environ.get("RORL_BENCH_ENCODER", "smamba_s32_c16_b2_nln")
ALGO = os.environ.get("RORL_BENCH_ALGO", "sac")
METRIC = "sac_update_trajectory_steps_per_s"


def model_kwargs(enc, value, hidden=None):
    hidden = hidden or (512 if enc.startswith("cgpt") else 256)      # SURVEY.md 8: encoder width 256 (cgpt: 512)
    return dict(state_dim=S_DIM, action_dim=A_DIM, embedding_size=128, embedding_hidden=[hidden, hidden],
                embedding_activations=['elu', 'elu', 'linear'], embedding_layer_type=['fc', enc, 'fc'],
                uni_model_hidden=[256, 256], uni_model_activations=['elu', 'elu', 'linear'],
                uni_model_layer_type=(['efc-8'] * 3 if value else ['fc'] * 3), fix_rnn_length=0,
                uni_model_input_mapping_dim=128, reward_input=False, last_action_input=True, last_state_input=True,
                separate_encoder=True)


HP = dict(gamma=0.99, sac_tau=0.995, policy_update_per=1, redq_m=2, policy_lr=3e-4, value_lr=1e-3, rnn_policy_lr=1e-5,
          rnn_value_lr=1e-5, alpha_lr=1e-4, target_entropy_ratio=1.0, sac_batch_size=N_TRAJ * T_LEN - 1,
          max_buffer_transition_num=N_TRAJ * T_LEN + 8)


def synth_trajectory(rng, T=T_LEN):
    """One trajectory in replay column order: state|last_state|last_action|action|next_state|reward|mask|start|done|
    reward_input|timeout  (SURVEY.md 8d 'Synthetic inputs')."""
    s = rng.standard_normal((T + 1, S_DIM))
    a = np.tanh(rng.standard_normal((T, A_DIM)))
    r = rng.standard_normal((T, 1))
    z = np.zeros
    last_s = np.vstack((z((1, S_DIM)), s[:T - 1]))
    last_a = np.vstack((z((1, A_DIM)), a[:T - 1]))
    r_in = np.vstack((z((1, 1)), r[:T - 1]))
    start = z((T, 1)); start[0] = 1
    done = z((T, 1)); done[-1] = 1
    return np.hstack((s[:T], last_s, last_a, a, s[1:], r, np.ones((T, 1)), start, done, r_in, done))


def template_transition():
    from rorl_b200.buffers.transition_buffer.replay_memory import Transition
    z = np.zeros
    return Transition(state=z((1, S_DIM)), last_state=z((1, S_DIM)), last_action=z((1, A_DIM)), action=z((1, A_DIM)),
                      next_state=z((1, S_DIM)), reward=0.0, logp=None, mask=1, done=False, timeout=False, start=True,
                      reward_input=z((1, 1)))


def workload_config(world):
    """`config` of the JSON line -- one function for both arms, so the reference arm reports the configuration it ran."""
    return {"workload": f"{ALGO.upper()} update, {ENCODER} encoder, {N_TRAJ} trajectories x {T_LEN} steps per GPU "
                        f"(obs {S_DIM}, act {A_DIM}, efc-8 twin-Q head, REDQ m=2, RESeL lr split)",
            "global_trajectories": N_TRAJ * world, "valid_steps_per_update": N_TRAJ * T_LEN * world,
            "parallelism": f"dp{world} (trajectory-sharded, NCCL grad all-reduce)" if world > 1 else "single GPU",
            "l2": "working set per step (activations > 1 GB) exceeds the 126 MB L2; no flush needed"}


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self._stop_evt = index, [], threading.Event()

    def run(self):
        while not self._stop_evt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip().split(",")
                self.samples.append([x.strip() for x in out])
            except Exception:
                pass
            self._stop_evt.wait(0.05)

    def summary(self):
        self._stop_evt.set()
        self.join(timeout=6)
        sm = [float(s[0]) for s in self.samples if len(s) >= 6 and s[0].replace('.', '').isdigit()]
        mx = [float(s[1]) for s in self.samples if len(s) >= 6 and s[1].replace('.', '').isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for s in self.samples if len(s) >= 6 for n, v in zip(names, s[2:6]) if v.lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist
    import rorl_b200._native as NV
    from rorl_b200.algorithm.sac_full_length_rnn_redq_sep_optim import SACFullLengthRNNREDQ_SEP_OPTIM
    from rorl_b200.algorithm.td3_full_length_rnn_redq_sep_optim import TD3FullLengthRNNREDQ_SEP_OPTIM

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    group = None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        group = dist.group.WORLD
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world}: launch N>1 with torch.distributed.run"
    torch.manual_seed(0)            # identical replicas on every rank
    np.random.seed(0)               # identical sampler / REDQ stream on every rank
    cls = SACFullLengthRNNREDQ_SEP_OPTIM if ALGO == "sac" else TD3FullLengthRNNREDQ_SEP_OPTIM
    alg = cls(dict(HP), model_kwargs(ENCODER, False), model_kwargs(ENCODER, True), T_LEN, device=dev, dist_group=group)
    alg.replay_buffer._init_memory_buffer(template_transition())
    rng = np.random.RandomState(1000 + rank)   # every rank owns different trajectories (trajectory sharding)
    for _ in range(N_TRAJ):
        alg.replay_buffer.push_trajectory_array(synth_trajectory(rng))
    torch.cuda.synchronize()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    # ---- device-resident arm -------------------------------------------------------------------------------------
    last = [None]

    def step_dev():
        last[0] = alg.train_one_batch(sync=False)
        return last[0]

    for _ in range(args.warmup):
        out = step_dev()
    valid_steps = out["real_batch_size"]
    clocks = ClockSampler(local) if rank == 0 else None
    if clocks:
        clocks.start()
    l0 = NV.launch_count()
    ms_total = timed(step_dev, args.steps)
    launches = NV.launch_count() - l0
    clk = clocks.summary() if clocks else None
    if args.dump_outputs and rank == 0:
        dump_outputs(alg, last[0], args.dump_outputs)
    ms_per_step = ms_total / args.steps
    value = valid_steps * world / (ms_per_step * 1e-3)

    # ---- end-to-end arm: host batch -> H2D -> update -> D2H scalars, every step -------------------------------------
    plan = alg.replay_buffer.plan_trajs(HP["sac_batch_size"], None, nest_stack_trajs=alg.allow_nest_stack)
    b_dev, v_dev = alg.replay_buffer.gather_device(plan)
    host_batch = b_dev.contiguous().cpu().pin_memory()
    host_valid = v_dev.contiguous().cpu().pin_memory()

    def step_e2e():
        res = alg.update_on_host_batch(host_batch, host_valid, plan.total_size, plan.lens, sync=True)
        assert np.isfinite(res["critic_loss"])

    for _ in range(args.warmup):          # >= 3: eager, graph capture, first replay
        step_e2e()
    e2e_steps = max(3, args.steps // 2)
    ms_e2e = timed(step_e2e, e2e_steps) / e2e_steps
    e2e = {"value": valid_steps * world / (ms_e2e * 1e-3), "unit": "trajectory-steps/s",
           "h2d_bytes_per_step": int(host_batch.numel() * 4 + host_valid.numel() * 4),
           "d2h_bytes_per_step": int(alg._stats.numel() * 4 + alg.Q_guard.state.numel() * 8 + 4), "ms_per_step": ms_e2e}

    # ---- strong-scaling leg (BASELINE config 5): 256 trajectories GLOBAL, 256 / N per GPU ------------------------------
    strong = None
    if not args.no_strong and STRONG_TRAJ % world == 0:
        n_local = STRONG_TRAJ // world
        hp_s = dict(HP, sac_batch_size=n_local * T_LEN - 1, max_buffer_transition_num=n_local * T_LEN + 8)
        torch.manual_seed(0)
        np.random.seed(0)
        alg_s = cls(hp_s, model_kwargs(ENCODER, False), model_kwargs(ENCODER, True), T_LEN, device=dev, dist_group=group)
        alg_s.replay_buffer._init_memory_buffer(template_transition())
        rng = np.random.RandomState(2000 + rank)
        for _ in range(n_local):
            alg_s.replay_buffer.push_trajectory_array(synth_trajectory(rng))
        step_s = lambda: alg_s.train_one_batch(sync=False)
        for _ in range(3):
            out_s = step_s()
        k_s = max(3, args.steps // 4)
        ms_s = timed(step_s, k_s) / k_s
        strong = {"scaling": "strong", "global_trajectories": STRONG_TRAJ, "trajectories_per_gpu": n_local, "steps": k_s,
                  "ms_per_step": ms_s, "value": out_s["real_batch_size"] * world / (ms_s * 1e-3), "unit": "trajectory-steps/s"}
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    line = {"metric": METRIC, "value": value, "unit": "trajectory-steps/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(world),
            "clocks": clk, "e2e": e2e, "gpu_launches": int(launches)}
    assert valid_steps == N_TRAJ * T_LEN
    if strong is not None:
        line["strong_scaling"] = strong
    if ENCODER.startswith("smamba"):
        line["roofline"] = scan_roofline(alg, dev, ms_per_step)
    line["roofline_gemm"] = gemm_roofline(dev)
    if world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline(encoder="gru", n_traj=N_TRAJ, updates=2, warm=1)
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


DUMP_BYTES = 63 << 20          # parameters + gradients; the small arrays stay well inside 64 MB in all


def dump_outputs(alg, out, path):
    """`--dump-outputs`: write what the last timed update computed as `path/<name>.npy` -- what `train_one_batch(sync=False)`
    returned (the device statistics vector and the host scalars) and the state it left: every parameter of the policy,
    critic and target critic and the gradients of the policy and critic (each model flattened in state_dict order), the
    entropy temperature and the Q-target guard.  The inputs are seeded, so two builds run with the same arguments can be
    compared array by array.  Should the parameters and gradients exceed DUMP_BYTES, every one of those arrays keeps
    every stride-th entry (the same fixed stride for all)."""
    import torch

    def flat(tensors):
        return torch.cat([t.detach().reshape(-1).float() for t in tensors]).cpu().numpy()

    arrays = {"stats_device": out["stats_device"].detach().cpu().numpy()}
    for k in ("real_batch_size", "real_batch_traj_num", "policy_updated"):
        arrays[k] = np.array(out[k], dtype=np.float64)
    for name, model in (("policy", alg.policy), ("value", alg.values[0]), ("target_value", alg.target_values[0])):
        arrays[f"{name}_params"] = flat(t for sd in model.state_dict().values() for t in sd.values())
    for name, model in (("policy", alg.policy), ("value", alg.values[0])):
        arrays[f"{name}_grads"] = flat(p.grad for m in model.contextual_modules.values() for p in m.parameters() if p.grad is not None)
    arrays["log_alpha"] = alg.log_sac_alpha.detach().cpu().numpy()
    arrays["q_guard"] = alg.Q_guard.state.detach().cpu().numpy()
    large = [k for k in arrays if k.endswith(("_params", "_grads"))]
    stride = -(-sum(arrays[k].nbytes for k in large) // DUMP_BYTES)
    os.makedirs(path, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(path, k + ".npy"), a[::stride] if k in large else a)


def scan_roofline(alg, dev, ms_per_step):
    """Time the selective-scan kernels alone at the workload shape [B=32, L=1019, D=512, N=32] (1000 steps + the replay's
    skip_step = d_conv + 2 blanks + 1, ref: nested_replay_memory.py:23,179) with CUDA events on the launch stream.
    Operands (4 x 66.8 MB) exceed L2, so consecutive launches do not hit in cache."""
    import torch
    import rorl_b200.kernels as K
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    B, L, D, Ns = N_TRAJ, T_LEN + 19, 512, 32
    g = torch.Generator(device=dev).manual_seed(0)
    rn = lambda *s: torch.randn(*s, device=dev, generator=g)
    u, delta, z = rn(B, L, D).requires_grad_(), (0.5 * rn(B, L, D) - 1).requires_grad_(), rn(B, L, D).requires_grad_()
    Bm, Cm = rn(B, L, Ns).requires_grad_(), rn(B, L, Ns).requires_grad_()
    A = (-torch.exp(0.3 * rn(D, Ns))).requires_grad_()
    Dk, bias = rn(D).requires_grad_(), rn(D).requires_grad_()
    start = torch.zeros(B, L, device=dev); start[:, :18] = 1
    dy = rn(B, L, D)

    def t(fn, n=20):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / n * 1e-3

    with torch.no_grad():
        t_fwd = t(lambda: K.selective_scan_tm(u, delta, A, Bm, Cm, Dk, z, bias, start, True))
    y = K.selective_scan_tm(u, delta, A, Bm, Cm, Dk, z, bias, start, True)
    t_both = t(lambda: torch.autograd.grad(K.selective_scan_tm(u, delta, A, Bm, Cm, Dk, z, bias, start, True), (u, delta, A, Bm, Cm, Dk, z, bias), dy), n=10)
    t_fwd_ck = t(lambda: K.selective_scan_tm(u, delta, A, Bm, Cm, Dk, z, bias, start, True), n=10)   # forward incl. checkpoints
    t_bwd = max(t_both - t_fwd_ck, 1e-9)
    bytes_fwd = 4 * (4 * B * D * L + 2 * B * Ns * L + B * L)            # SURVEY.md 8d
    bytes_bwd = 4 * (7 * B * D * L + 4 * B * Ns * L)
    # per update: 2 blocks x (5 forward, 2 backward) launches
    share_fwd, share_bwd = 10 * t_fwd / (ms_per_step * 1e-3), 4 * t_bwd / (ms_per_step * 1e-3)
    if share_bwd > share_fwd:
        name, ach, alg_bytes = "selscan_bwd_kernel<32>", bytes_bwd / t_bwd / 1e9, bytes_bwd
    else:
        name, ach, alg_bytes = "selscan_fwd_kernel<32>", bytes_fwd / t_fwd / 1e9, bytes_fwd
    # DRAM traffic per launch of that kernel from the committed ncu --set full capture (profiles/): not measurable live
    traffic, xu = None, None
    try:
        cap = json.load(open(os.path.join(ROOT, "profiles", "selscan_ncu_traffic.json")))[name]
        traffic, xu = cap["dram_bytes_read"] + cap["dram_bytes_write"], cap.get("xu_pipe_pct")
    except Exception:
        pass
    return {"bound": "hbm", "kernel": name, "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
            "traffic": traffic, "traffic_source": "profiles/selscan_ncu_traffic.json (ncu --set full, same shape)",
            "xu_pipe_pct_ncu": xu,
            "algorithmic_bytes_per_launch": alg_bytes, "peak_source": "MEASURED_PEAKS.json hbm_gbs (burst copy)" if peaks else "fallback 6650 GB/s",
            "fwd": {"us": t_fwd * 1e6, "GBps": bytes_fwd / t_fwd / 1e9, "share_of_step": share_fwd},
            "bwd": {"us": t_bwd * 1e6, "GBps": bytes_bwd / t_bwd / 1e9, "share_of_step": share_bwd},
            "note": "selective scan at d_state=32 is MUFU/FMA-pipe bound, not HBM bound (SURVEY.md App. F)"}


def gemm_roofline(dev):
    """Second roofline object, for the kernel with the largest share of the step (the tcgen05 GEMM, ~39 %): the
    in_proj-half shape [32608, 256] x [512, 256]^T timed alone with CUDA events.  `achieved` counts the useful fp32 FLOPs
    (2 M N K); the kernel issues three bf16 MMAs for them (two-term bf16 split, csrc/gemm_bf16.cu).  `peak` is the
    measured dense bf16 rate of MEASURED_PEAKS.json."""
    import torch
    import rorl_b200.kernels as K
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        peaks = {}
    peak = float(peaks.get("bf16_tflops", 1590.0))
    M, Nn, Kk = N_TRAJ * (T_LEN + 19), 512, 256
    g = torch.Generator(device=dev).manual_seed(1)
    a = torch.randn(M, Kk, device=dev, generator=g)
    w = torch.randn(Nn, Kk, device=dev, generator=g)
    for _ in range(3):
        K.gemm_tn(a, w)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(20):
        K.gemm_tn(a, w)
    e1.record()
    torch.cuda.synchronize()
    t = e0.elapsed_time(e1) / 20 * 1e-3
    useful = 2.0 * M * Nn * Kk
    ncu = {}
    try:
        for row in json.load(open(os.path.join(ROOT, "profiles", "r02_ncu_summary.json"))):
            if row["kernel"].startswith("void gemm_bf16x3_kernel<256, 0>") and abs(row.get("us", 0) - 41.0) < 3:
                ncu = row
    except Exception:
        pass
    return {"bound": "tensor", "kernel": "gemm_bf16x3_kernel<BN 256, TN> (two-term bf16 split: 3 MMAs on kind::f16; includes the B pre-split launch)",
            "shape": [M, Nn, Kk], "us": t * 1e6, "achieved": useful / t / 1e12, "issued_bf16": 3 * useful / t / 1e12, "peak": peak,
            "unit": "TFLOP/s", "frac": useful / t / 1e12 / peak, "frac_issued_of_bf16_peak": 3 * useful / t / 1e12 / peak,
            "peak_source": "MEASURED_PEAKS.json bf16_tflops (burst)" if peaks else "fallback 1590 TFLOP/s bf16",
            "tensor_pipe_pct_ncu": ncu.get("tensor_pipe_cycles_pct"), "l1tex_pct_ncu": ncu.get("l1tex_pct"),
            "ncu_source": "profiles/r02_ncu_summary.json (same shape, ncu --set full)"}


# ------------------------------------------------------------------------------------------------------------------
def oracle_update_runner(encoder, n_traj, algo="sac", s_dim=None, a_dim=None, t_len=None):
    """Build the oracle's CPU update (test infrastructure; allowed here as the cpu_baseline / reference leg)."""
    import torch
    from oracle import model as OM, sampler as OS, update as OU
    from rorl_b200.policy_value_models.make_models import make_policy_model, make_value_model
    global S_DIM, A_DIM, T_LEN
    saved = (S_DIM, A_DIM, T_LEN)
    S_DIM, A_DIM, T_LEN = s_dim or S_DIM, a_dim or A_DIM, t_len or T_LEN
    try:
        return _oracle_update_runner(encoder, n_traj, algo, OM, OS, OU, make_policy_model, make_value_model, torch)
    finally:
        S_DIM, A_DIM, T_LEN = saved


def _oracle_update_runner(encoder, n_traj, algo, OM, OS, OU, make_policy_model, make_value_model, torch):
    torch.manual_seed(0)
    np.random.seed(0)
    pk, vk = model_kwargs(encoder, False), model_kwargs(encoder, True)
    pol, val = make_policy_model(pk, algo, False), make_value_model(vk, algo, False)   # weights only (CPU tensors)
    skip = 1 + max([l.d_conv for l in pol.embedding_network.layer_list if hasattr(l, 'd_conv')] + [0])
    buf = OS.RefNestedReplay(n_traj * T_LEN + 8, T_LEN, additional_history_len=skip)
    rng = np.random.RandomState(1000)
    for _ in range(n_traj):
        rows = synth_trajectory(rng, T_LEN)
        if buf.buf is None:
            t = template_transition()
            buf._init(t)
        n = rows.shape[0]
        buf.traj_start.append(buf.ptr)
        buf.buf[buf.ptr:buf.ptr + n] = rows
        buf.ptr += n
        buf.traj_len.append(n)
        buf.count += n
    hp = dict(HP, sac_batch_size=n_traj * T_LEN - 1, sample_std=0.1, target_action_noise_std=0.04, target_action_noise_clip=0.12)
    gen = torch.Generator().manual_seed(1)
    upd = OU.RefUpdate(pol.state_dict(), val.state_dict(), OM.ModelSpec(**pk), OM.ModelSpec(**vk), hp, buf,
                       lambda shape: torch.randn(shape, generator=gen), algo=algo, redq=True,
                       allow_nest_stack=('gru' not in encoder))
    return upd, n_traj * T_LEN


def reference_update_runner(encoder, n_traj, algo="sac", s_dim=None, a_dim=None, t_len=None, t_cut=None):
    """The UNMODIFIED reference's algorithm object on CPU (oracle/refload.py harness over /root/reference or the staged
    oracle/_ref copy), replay filled through its own `mem_push` with `n_traj` synthetic trajectories of `t_cut or t_len`
    steps.  Returns (object with .train_one_batch(), valid steps per update) or None if the reference is not available."""
    from oracle import refload
    if not refload.available():
        return None
    import torch
    refload.load_reference(gpu_semantics=False)       # the reference as it runs on a CPU-only machine
    refload.install_algo_stubs()
    from offpolicy_rnn.buffers.transition_buffer.replay_memory import Transition
    global S_DIM, A_DIM, T_LEN
    saved = (S_DIM, A_DIM, T_LEN)
    S_DIM, A_DIM, T_LEN = s_dim or S_DIM, a_dim or A_DIM, t_len or T_LEN
    try:
        torch.manual_seed(0)
        np.random.seed(0)
        steps = t_cut or T_LEN
        hp = dict(refload.REF_HP, sac_batch_size=n_traj * steps - 1, max_buffer_transition_num=n_traj * steps + 8)
        cls = "SACFullLengthRNNREDQ_SEP_OPTIM" if algo == "sac" else "TD3FullLengthRNNREDQ_SEP_OPTIM"
        A = refload.build_algorithm(cls, hp, model_kwargs(encoder, False), model_kwargs(encoder, True), T_LEN, A_DIM)
        rng = np.random.RandomState(1000)
        S, Ad = S_DIM, A_DIM
        for _ in range(n_traj):
            rows = synth_trajectory(rng, T_LEN)[:steps]
            for t in range(steps):
                r = rows[t]
                last = t == steps - 1
                A.replay_buffer.mem_push(Transition(
                    state=r[None, 0:S], last_state=r[None, S:2 * S], last_action=r[None, 2 * S:2 * S + Ad],
                    action=r[None, 2 * S + Ad:2 * S + 2 * Ad], next_state=r[None, 2 * S + 2 * Ad:3 * S + 2 * Ad],
                    reward=float(r[3 * S + 2 * Ad]), logp=None, mask=1, done=last, timeout=last, start=(t == 0),
                    reward_input=r[None, 3 * S + 2 * Ad + 4:3 * S + 2 * Ad + 5]))

        class Runner:
            def train_one_batch(self_inner):
                out = A.train_one_batch()
                A.grad_num += 1
                return out
        return Runner(), n_traj * steps
    finally:
        S_DIM, A_DIM, T_LEN = saved


def _time_updates(upd, updates, warm):
    for _ in range(warm):
        upd.train_one_batch()
    t0 = time.perf_counter()
    for _ in range(updates):
        upd.train_one_batch()
    return (time.perf_counter() - t0) / updates


def cpu_baseline(encoder, n_traj, updates, warm):
    """The reference's CPU path (GRU encoder, north_star) on this box's host cores: the reference's own code when the
    staged copy is present (kind "reference"), else the oracle port (kind "port")."""
    import torch
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    built = reference_update_runner(encoder, n_traj)
    kind = "reference" if built is not None else "port"
    upd, valid = built if built is not None else oracle_update_runner(encoder, n_traj)
    what = "the reference's own train_one_batch (SACFullLengthRNNREDQ_SEP_OPTIM, unmodified code from oracle/_ref)" \
        if kind == "reference" else "the oracle CPU port"
    dt = _time_updates(upd, updates, warm)
    out = {"value": valid / dt, "unit": "trajectory-steps/s", "cores": cores, "kind": kind,
           "sample": f"{updates} timed SAC updates (after {warm} warm-up) of {what} with the {encoder} encoder on "
                     f"{n_traj} trajectories x {T_LEN} steps, torch CPU ops on {cores} threads", "s_per_update": dt}
    # the reference's own CPU-runnable case (BASELINE.json configs[0]): Pendulum-V shapes, 8 trajectories x 200 steps
    built = reference_update_runner(encoder, 8, s_dim=1, a_dim=1, t_len=200)
    upd, valid = built if built is not None else oracle_update_runner(encoder, 8, s_dim=1, a_dim=1, t_len=200)
    dt1 = _time_updates(upd, 3, 1)
    out["config1"] = {"value": valid / dt1, "unit": "trajectory-steps/s", "s_per_update": dt1, "kind": kind,
                      "sample": f"3 timed SAC updates (after 1 warm-up), {encoder} encoder, 8 trajectories x 200 steps, obs 1, act 1"}
    return out


def run_reference(args):
    """Reference arm: the reference's own CPU implementation of this arm's configuration (see the module docstring) on
    all host threads.  Rank 0 only; the other ranks exit without work."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    import torch
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    t_cut = int(os.environ.get("RORL_REF_TLEN", "100"))
    built = reference_update_runner(ENCODER, N_TRAJ, ALGO, t_cut=t_cut)
    kind = "reference" if built is not None else "port"
    if built is None:                                   # staged copy missing: time the oracle port on the same sample
        upd, valid = oracle_update_runner(ENCODER, N_TRAJ, ALGO, t_len=t_cut)
    else:
        upd, valid = built
    dt = _time_updates(upd, args.steps, args.warmup)
    v = valid / dt
    impl = ("the reference's own train_one_batch, unmodified code staged under oracle/_ref, as it runs on a CPU-only machine "
            "(smamba: per-time-step Mamba.step loop, ref smamba/mamba.py:133-159)") if kind == "reference" else "the oracle CPU port"
    sample = (f"each step = one full {ALGO.upper()} update of {impl} with the {ENCODER} encoder on {N_TRAJ} trajectories cut to "
              f"{t_cut} of their {T_LEN} steps ({valid} valid steps; the loop over time is linear in the length, the {N_TRAJ} rows "
              f"it amortises over are the workload's), {cores} host threads")
    print(json.dumps({"impl": "reference", "metric": METRIC, "value": v, "unit": "trajectory-steps/s", "n_gpus": args.gpus,
                      "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
                      "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                      "config": workload_config(args.gpus),
                      "cpu_baseline": {"value": v, "unit": "trajectory-steps/s", "cores": cores, "kind": kind, "sample": sample},
                      "e2e": {"value": v, "unit": "trajectory-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=None)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-strong", action="store_true", help="skip the 256-trajectory strong-scaling leg")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed update computed to DIR/<name>.npy")
    a = ap.parse_args()
    if a.steps is not None and a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    if a.impl == "reference":
        a.steps = a.steps if a.steps is not None else 3
        a.warmup = a.warmup if a.warmup is not None else 1
        run_reference(a)
    else:
        a.steps = a.steps if a.steps is not None else 50        # ~1 s timed region: several nvidia-smi clock samples
        a.warmup = max(3, a.warmup if a.warmup is not None else 3)
        run_ours(a)
