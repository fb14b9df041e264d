#!/usr/bin/env python
"""Time the discrete-action SAC update: one JSON line per case.

    python tools/bench_discrete.py [--steps K] [--warmup W] [--only SUBSTRING]

Workload: 32 trajectories x 1000 steps of a synthetic discrete-action replay (obs 9, A actions; the action is the index,
the last action its one-hot), width 256 as in bench.py, efc-8 Q head, fixed alpha 0.2.  Cases: encoders gilr and
smamba_s32_c16_b2_nln, A = 4 and 18, the REDQ class (target min over m = 2 members, actor mean) and the ensembleQ class
(min over all 8).  The ensembleQ classes hand the target policy the raw action index as its last action (ref:
sac_full_length_rnn_ensembleQ.py:141), which only fits a policy without last-action input, so those cases run with
last_action_input=False.  Timing as in bench.py: `train_one_batch(sync=False)` with the replay resident in HBM, CUDA events
around K updates after W warm-up updates (from the third update on, the update is replayed from captured CUDA graphs).
The card's name and power limit are part of every line.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

S_DIM, T_LEN, N_TRAJ, WIDTH = 9, 1000, 32, 256
ENCODERS = ("gilr", "smamba_s32_c16_b2_nln")
ACTIONS = (4, 18)
CLASSES = {"redq": "sac_rnn_full_horizon_redQ_sep_optim", "ensembleq": "sac_rnn_full_horizon_ensemble_q_sep_optim"}


def model_kwargs(enc, A, value, last_action):
    return dict(state_dim=S_DIM, action_dim=A, embedding_size=128, embedding_hidden=[WIDTH, WIDTH],
                embedding_activations=['elu', 'elu', 'linear'], embedding_layer_type=['fc', enc, 'fc'],
                uni_model_hidden=[256, 256], uni_model_activations=['elu', 'elu', 'linear'],
                uni_model_layer_type=(['efc-8'] * 3 if value else ['fc'] * 3), fix_rnn_length=0,
                uni_model_input_mapping_dim=128, reward_input=False, last_action_input=last_action, last_state_input=True,
                separate_encoder=True)


HP = dict(gamma=0.99, sac_tau=0.995, policy_update_per=1, redq_m=2, policy_lr=3e-4, value_lr=1e-3, rnn_policy_lr=1e-5,
          rnn_value_lr=1e-5, alpha_lr=1e-4, target_entropy_ratio=1.0, sac_alpha=0.2, sac_batch_size=N_TRAJ * T_LEN - 1,
          max_buffer_transition_num=N_TRAJ * T_LEN + 8)


def synth_trajectory(rng, A, T=T_LEN):
    """Replay column order: state|last_state|last_action (one-hot)|action (index)|next_state|reward|mask|start|done|
    reward_input|timeout."""
    s = rng.standard_normal((T + 1, S_DIM))
    a = rng.randint(A, size=T)
    onehot = np.eye(A)[a]
    r = rng.standard_normal((T, 1))
    z = np.zeros
    last_s = np.vstack((z((1, S_DIM)), s[:T - 1]))
    last_a = np.vstack((z((1, A)), onehot[:T - 1]))
    r_in = np.vstack((z((1, 1)), r[:T - 1]))
    start = z((T, 1)); start[0] = 1
    done = z((T, 1)); done[-1] = 1
    return np.hstack((s[:T], last_s, last_a, a[:, None].astype(np.float64), s[1:], r, np.ones((T, 1)), start, done, r_in, done))


def template_transition(A):
    from rorl_b200.buffers.transition_buffer.replay_memory import Transition
    z = np.zeros
    return Transition(state=z((1, S_DIM)), last_state=z((1, S_DIM)), last_action=z((1, A)), action=z((1, 1)),
                      next_state=z((1, S_DIM)), reward=0.0, logp=None, mask=1, done=False, timeout=False, start=True,
                      reward_input=z((1, 1)))


def card():
    import torch
    out = {"gpu": torch.cuda.get_device_name(0), "power_limit_w": None}
    try:
        q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=power.limit", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=10).stdout.strip()
        out["power_limit_w"] = float(q)
    except Exception:
        pass
    return out


def run_case(enc, A, kind, steps, warmup, dev):
    import torch
    from rorl_b200.utility.alg_init import alg_class
    torch.manual_seed(0)
    np.random.seed(0)
    last_action = kind == "redq"
    alg = alg_class(CLASSES[kind])(dict(HP), model_kwargs(enc, A, False, last_action), model_kwargs(enc, A, True, last_action),
                                   T_LEN, device=dev, discrete_env=True)
    alg.replay_buffer._init_memory_buffer(template_transition(A))
    rng = np.random.RandomState(1000)
    for _ in range(N_TRAJ):
        alg.replay_buffer.push_trajectory_array(synth_trajectory(rng, A))
    step = lambda: alg.train_one_batch(sync=False)
    for _ in range(warmup):
        out = step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        out = step()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    stats = out["stats_device"].tolist()
    assert np.isfinite(stats[2]) and np.isfinite(stats[4]), stats
    return {"metric": "sac_discrete_update_ms_per_step", "encoder": enc, "action_dim": A, "class": kind,
            "trajectories": N_TRAJ, "steps_per_trajectory": T_LEN, "width": WIDTH, "ms_per_step": ms,
            "trajectory_steps_per_s": out["real_batch_size"] / (ms * 1e-3), "timed_updates": steps, "warmup": warmup,
            "graph_segments_captured": sum(isinstance(v, dict) for v in getattr(alg, "_graphs", {}).values()),
            "side_stream": getattr(alg, "_side_stream", None) is not None,
            "critic_loss": stats[2], "actor_loss": stats[4]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--only", default="", help="run the cases whose '<encoder>/<A>/<class>' contains this")
    args = ap.parse_args()
    import torch
    dev = torch.device("cuda", 0)
    info = card()
    for enc in ENCODERS:
        for A in ACTIONS:
            for kind in CLASSES:
                if args.only not in f"{enc}/{A}/{kind}":
                    continue
                line = run_case(enc, A, kind, args.steps, args.warmup, dev)
                line.update(info)
                print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
