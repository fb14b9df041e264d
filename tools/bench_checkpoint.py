"""Wall time of saving and restoring the update engine's full state (`state_dict()` + `torch.save`,
`torch.load(weights_only=True)` + `load_state_dict()`), at the benchmark's shape (SAC + smamba_s32_c16_b2_nln, width 256,
32 trajectories x 1000 steps in the replay) and with a filled 10^6-transition replay (1000 x 1000 steps).

    python tools/bench_checkpoint.py [--repeats R] [--out FILE]

Each case runs a few updates first (graphs captured, optimizer state non-trivial), then times R save / load pairs with
a host clock; every timed region ends in a device synchronise.  The checkpoint goes to a temporary directory (page
cache: the times do not include the disk flush).  Prints one JSON line per case, with the GPU name and power limit.
"""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_card():
    try:
        return subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=10).stdout.strip()
    except Exception as e:  # noqa: BLE001
        return f"unavailable ({e})"


def run_case(name, n_traj, capacity, repeats, tmp):
    import torch
    import bench as B
    from rorl_b200.algorithm.sac_full_length_rnn_redq_sep_optim import SACFullLengthRNNREDQ_SEP_OPTIM
    dev = torch.device("cuda", 0)
    torch.manual_seed(0)
    np.random.seed(0)
    hp = dict(B.HP, max_buffer_transition_num=capacity)
    alg = SACFullLengthRNNREDQ_SEP_OPTIM(hp, B.model_kwargs(B.ENCODER, False), B.model_kwargs(B.ENCODER, True), B.T_LEN, device=dev)
    alg.replay_buffer._init_memory_buffer(B.template_transition())
    rng = np.random.RandomState(1000)
    for _ in range(n_traj):
        alg.replay_buffer.push_trajectory_array(B.synth_trajectory(rng))
    for _ in range(3):
        alg.train_one_batch()
    torch.cuda.synchronize(dev)
    path = os.path.join(tmp, f"{name}.pt")
    save_s, load_s = [], []
    for _ in range(repeats):
        t0 = time.perf_counter()
        torch.save(alg.state_dict(), path)
        save_s.append(time.perf_counter() - t0)
        t0 = time.perf_counter()
        alg.load_state_dict(torch.load(path, weights_only=True))
        torch.cuda.synchronize(dev)
        load_s.append(time.perf_counter() - t0)
    size = os.path.getsize(path)
    log = alg.train_one_batch()               # the engine still trains after the loads
    assert np.isfinite(log["critic_loss"])
    del alg
    torch.cuda.empty_cache()
    return {"case": name, "encoder": B.ENCODER, "replay_transitions": n_traj * B.T_LEN, "replay_capacity": capacity,
            "file_mb": round(size / 2 ** 20, 1), "save_s": [round(x, 3) for x in save_s], "load_s": [round(x, 3) for x in load_s],
            "save_median_s": round(float(np.median(save_s)), 3), "load_median_s": round(float(np.median(load_s)), 3)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_checkpoint needs a CUDA device")
    card = gpu_card()
    tmp = tempfile.mkdtemp(prefix="rorl_ckpt_")
    rows = []
    try:
        for name, n_traj, cap in (("bench_shape", 32, 32 * 1000 + 8), ("replay_1e6", 1000, 1000000)):
            r = dict(run_case(name, n_traj, cap, args.repeats, tmp), gpu=card)
            print(json.dumps(r), flush=True)
            rows.append(r)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    if args.out:
        with open(args.out, "w") as f:
            for r in rows:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
