"""Exact resume: a run stopped after k updates, saved with `state_dict()` + `torch.save` and continued in a fresh engine
from `torch.load(weights_only=True)` + `load_state_dict()`, must log and leave what a run that never stopped logs and
leaves.  Also: rewinding a live engine with captured CUDA graphs, refusal of mismatched checkpoints, data parallel."""
import os
import sys

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

from test_update_gpu import fill_buffer, fill_buffer_discrete

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEV = torch.device("cuda:0")
S, A, H = 5, 3, 64
LENS = [40, 40, 40, 40]
K_STEPS = 3                    # updates before the save, and after it

# name -> (algorithm, encoder, discrete, extra hyper-parameters)
CASES = {
    # value-norm + embedding value clipping (smamba A_log at 1e-3) and weight decay (the frozen set)
    "sac_redq_sep_smamba": ("sac_rnn_full_horizon_redQ_sep_optim", "smamba_s16_c4_b1", False,
                            dict(value_max_gradnorm=1.0, value_embedding_max_gradnorm=0.5, policy_embedding_max_gradnorm=0.5,
                                 policy_l2_norm=1e-3)),
    "td3_ensembleq_gilr": ("td3_rnn_full_horizon_ensembleQ", "gilr", False, {}),
    "sac_discrete_gru": ("sac_rnn_full_horizon_redQ_sep_optim", "gru", True, dict(policy_update_per=2, sac_alpha=0.2)),
    "sac_lstm_rndhidden": ("sac_rnn_full_horizon_redQ", "lstm", False, dict(randomize_first_hidden=True)),
    "sac_lru_utd2": ("sac_rnn_full_horizon_redQ", "lru", False, dict(utd=2)),
    "sac_cgpt": ("sac_rnn_full_horizon_redQ_sep_optim", "cgpt_h2_l1_p0.1", False, {}),
}


def _kw(enc, value, width=H, ensemble=8):
    return dict(state_dim=S, action_dim=A, embedding_size=32, embedding_hidden=[width, width],
                embedding_activations=['elu', 'elu', 'linear'], embedding_layer_type=['fc', enc, 'fc'], uni_model_hidden=[width, width],
                uni_model_activations=['elu', 'elu', 'linear'],
                uni_model_layer_type=([f'efc-{ensemble}'] * 3 if value else ['fc'] * 3), fix_rnn_length=0,
                uni_model_input_mapping_dim=32, reward_input=False, last_action_input=True, last_state_input=True,
                separate_encoder=True)


def _hp(**kw):
    return dict(dict(gamma=0.99, sac_tau=0.995, policy_update_per=1, redq_m=2, policy_lr=3e-4, value_lr=1e-3, rnn_policy_lr=1e-5,
                     rnn_value_lr=1e-5, alpha_lr=1e-4, target_entropy_ratio=1.0, sac_batch_size=sum(LENS) - 1,
                     max_buffer_transition_num=1000), **kw)


def _engine(case, graph, seed, fill=True, enc=None, width=H, ensemble=8, discrete=None, dist_group=None, device=DEV):
    from rorl_b200.buffers.transition_buffer.replay_memory import Transition
    from rorl_b200.utility.alg_init import alg_class
    name, enc0, disc0, extra = CASES[case]
    enc = enc or enc0
    disc = disc0 if discrete is None else discrete
    torch.manual_seed(seed)
    np.random.seed(seed)
    alg = alg_class(name)(_hp(use_cuda_graph=graph, **extra), _kw(enc, False, width), _kw(enc, True, width, ensemble), max(LENS),
                          device=device, discrete_env=disc, dist_group=dist_group)
    if fill:
        (fill_buffer_discrete if disc else fill_buffer)(alg.replay_buffer, Transition, np.random.RandomState(4), LENS, S, A)
        np.random.seed(50)
    return alg


def _state(alg):
    """Every tensor the resumed run must reproduce."""
    out = {}
    for tag, model in (("p", alg.policy), ("v", alg.values[0]), ("t", alg.target_values[0]), ("tp", alg.target_policy)):
        for m, params in model.state_dict().items():
            for n, t in params.items():
                out[f"{tag}/{m}/{n}"] = t.detach().clone()
    for tag, opt in (("pol", alg.optimizer_policy), ("val", alg.optimizer_value), ("alpha", alg.optimizer_alpha)):
        out[f"{tag}/m"], out[f"{tag}/v"], out[f"{tag}/step"] = opt.m.clone(), opt.v.clone(), opt.step_count.clone()
    out["log_alpha"] = alg.log_sac_alpha.detach().clone()
    out["guard"] = alg.Q_guard.state.clone()
    return out


def _save_load(alg, path):
    torch.save(alg.state_dict(), path)
    return torch.load(path, weights_only=True)


def _fresh_instances(monkeypatch):
    from rorl_b200.models.flash_attention.TransformerFlashAttention import MHA
    monkeypatch.setattr(MHA, "_instances", 0)           # the straight and the saved run draw the same dropout salts


def _straight_and_resumed(case, graph, tmp_path, monkeypatch):
    _fresh_instances(monkeypatch)
    a = _engine(case, graph, 3)
    logs_a = [a.train_one_batch() for _ in range(2 * K_STEPS)]
    state_a = _state(a)
    _fresh_instances(monkeypatch)
    b = _engine(case, graph, 3)
    for _ in range(K_STEPS):
        b.train_one_batch()
    path = str(tmp_path / "ckpt.pt")
    torch.save(b.state_dict(), path)
    del b
    # a fresh engine under other seeds, built after the others (other cgpt dropout salts), with an empty replay buffer
    c = _engine(case, graph, 11, fill=False)
    np.random.seed(12)
    c.load_state_dict(torch.load(path, weights_only=True))
    logs_c = [c.train_one_batch() for _ in range(K_STEPS)]
    return logs_a[K_STEPS:], logs_c, state_a, _state(c), a


@pytest.mark.parametrize("case", list(CASES))
def test_resumed_run_equals_straight_run_eager(case, tmp_path, monkeypatch):
    logs_a, logs_c, sa, sc, _ = _straight_and_resumed(case, False, tmp_path, monkeypatch)
    for i, (la, lc) in enumerate(zip(logs_a, logs_c)):
        assert la == lc, (i, {k: (la[k], lc.get(k)) for k in la if la[k] != lc.get(k)})
    for k in sa:
        assert torch.equal(sa[k], sc[k]), k


@pytest.mark.parametrize("case", list(CASES))
def test_resumed_run_equals_straight_run_with_graphs(case, tmp_path, monkeypatch):
    """With CUDA graphs on, the straight run replays a graph where the resumed engine's first update is eager (and its
    second is captured).  test_cuda_graph_replay_matches_eager allows rounding-level differences between eager and
    replayed launches, because the cuBLAS calls left on the path (K < 32 projections) could pick another algorithm
    under capture.  At these shapes they do not: replayed and eager updates leave the same bits on a B200, so the
    resumed run is held to bit identity here too, CUDA random draws included."""
    logs_a, logs_c, sa, sc, a = _straight_and_resumed(case, True, tmp_path, monkeypatch)
    assert any(isinstance(v, dict) for v in a._graphs.values()), "no graph was captured"
    for i, (la, lc) in enumerate(zip(logs_a, logs_c)):
        assert la == lc, (i, {k: (la[k], lc.get(k)) for k in la if la[k] != lc.get(k)})
    for k in sa:
        assert torch.equal(sa[k], sc[k]), k


@pytest.mark.parametrize("case", ["sac_redq_sep_smamba", "sac_cgpt", "sac_discrete_gru"])
def test_rewind_live_engine_with_graphs(case, tmp_path, monkeypatch):
    """Load a saved state back into the same engine after it has captured and replayed graphs: the graphs read the
    restored tensors (the load copies in place and keeps them), so the second pass repeats the first bit for bit."""
    alg = _engine(case, True, 3)
    for _ in range(K_STEPS):
        alg.train_one_batch()
    assert any(isinstance(v, dict) for v in alg._graphs.values()), "no graph was captured"
    sd = _save_load(alg, str(tmp_path / "rewind.pt"))
    passes = []
    for _ in range(2):
        logs = [alg.train_one_batch() for _ in range(K_STEPS)]
        passes.append((logs, _state(alg)))
        graphs = [id(v) for v in alg._graphs.values() if isinstance(v, dict)]
        alg.load_state_dict(sd)
        assert [id(v) for v in alg._graphs.values() if isinstance(v, dict)] == graphs, "the load dropped the graphs"
    (l1, s1), (l2, s2) = passes
    assert l1 == l2
    for k in s1:
        assert torch.equal(s1[k], s2[k]), k


@pytest.mark.parametrize("what,field", [("encoder", "policy.embedding_layer_type"), ("width", "policy.embedding_hidden"),
                                        ("ensemble", "ensemble_size"), ("discrete", "discrete_env"), ("format", "format")])
def test_mismatched_checkpoint_is_refused(what, field, tmp_path):
    src = _engine("sac_redq_sep_smamba", False, 3)
    src.train_one_batch()
    sd = _save_load(src, str(tmp_path / "src.pt"))
    kw = {"encoder": dict(enc="gilr"), "width": dict(width=128), "ensemble": dict(ensemble=4), "discrete": dict(discrete=True),
          "format": {}}[what]
    if what == "format":
        sd = dict(sd, format=sd["format"] + 1)
    dst = _engine("sac_redq_sep_smamba", False, 5, **kw)
    dst.train_one_batch()
    before = _state(dst)
    buf = (list(dst.replay_buffer.trajectory_start), dst.replay_buffer.ptr, dst.grad_num)
    with pytest.raises(ValueError, match=field.replace(".", r"\.")):
        dst.load_state_dict(sd)
    after = _state(dst)
    for k in before:
        assert torch.equal(before[k], after[k]), k
    assert buf == (list(dst.replay_buffer.trajectory_start), dst.replay_buffer.ptr, dst.grad_num)
    log = dst.train_one_batch()
    assert np.isfinite(log["critic_loss"])


def test_weights_part_loads_with_load_models(tmp_path):
    """The `policy` / `value` entries are the reference's state_dict layout: `load_models` takes them as they are."""
    a = _engine("td3_ensembleq_gilr", False, 3)
    a.train_one_batch()
    sd = _save_load(a, str(tmp_path / "w.pt"))
    b = _engine("td3_ensembleq_gilr", False, 7)
    b.load_models(sd["policy"], sd["value"])
    for (ka, ta), (kb, tb) in zip(_state(a).items(), _state(b).items()):
        if ka.startswith(("p/", "v/")):
            assert torch.equal(ta, tb), ka


# ---- data parallel ------------------------------------------------------------------------------------------------------
def _dp_run(rank, world, port, mode, out):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import torch.distributed as dist
    from rorl_b200.buffers.transition_buffer.replay_memory import Transition
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    fresh = mode == "resume"
    alg = _engine("sac_redq_sep_smamba", False, 11 if fresh else 3, fill=False, dist_group=dist.group.WORLD, device=dev)
    if not fresh:
        fill_buffer(alg.replay_buffer, Transition, np.random.RandomState(4 + rank), LENS, S, A)
        np.random.seed(50)
    else:
        alg.load_state_dict(torch.load(f"{out}.ckpt.{rank}", weights_only=True))
    n = 2 * K_STEPS if mode == "straight" else K_STEPS
    logs = [alg.train_one_batch() for _ in range(n)]
    if mode == "save":
        torch.save(alg.state_dict(), f"{out}.ckpt.{rank}")
    else:
        torch.save({"logs": logs[-K_STEPS:], "state": {k: v.cpu() for k, v in _state(alg).items()}}, f"{out}.{mode}.{rank}")
    dist.destroy_process_group()


def test_data_parallel_resume(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    out = str(tmp_path / "dp")
    port = 29800 + os.getpid() % 1000
    for i, mode in enumerate(("straight", "save", "resume")):
        mp.start_processes(_dp_run, args=(2, port + i, mode, out), nprocs=2, join=True, start_method="spawn")
    for r in range(2):
        a, c = torch.load(f"{out}.straight.{r}"), torch.load(f"{out}.resume.{r}")
        assert a["logs"] == c["logs"], r
        for k in a["state"]:
            assert torch.equal(a["state"][k], c["state"][k]), (r, k)
