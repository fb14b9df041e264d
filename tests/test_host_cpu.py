"""Host-side logic that needs no GPU: the C-ABI library loads and exports every declared symbol, the layer
registry / state_dict / RESeL split are compatible with the reference, and the sampler's integer plan
reproduces the reference batches bit for bit (plan applied with numpy here, with the CUDA gather on the GPU)."""
import ctypes
import os

import numpy as np
import pytest
import torch

from helpers import cfg_of, load_npz, nested_sd


def test_library_exports_every_declared_symbol():
    import rorl_b200._native as N
    assert os.path.exists(N.LIB_PATH), "build the library first: python -c 'import __graft_entry__ as g; g.build()'"
    lib = ctypes.CDLL(N.LIB_PATH)
    protos = N.declared_prototypes()
    assert len(protos) >= 25
    missing = [n for n in protos if not hasattr(lib, n)]
    assert not missing, missing
    assert N.lib().rorl_abi_version() == 6
    assert N.lib().rorl_selscan_dtile(32) == 64 and N.lib().rorl_selscan_dtile(7) < 0


def test_gemm_abi_takes_bf16_passes_only():
    """rorl_gemm_tn / rorl_gemm_nt take passes 2 and 4 only and refuse any other value before any CUDA call; the split
    copy of B has rows padded to a multiple of 8 bf16; the tile / k-depth / debug switches are gone."""
    import rorl_b200._native as N
    L, d = N.lib(), 4096                              # never dereferenced
    for passes in (1, 3):
        assert L.rorl_gemm_tn(d, d, None, d, None, 128, 128, 64, 1, 64, 64, 128, 0, 0, 0, 0, 0, passes, 0, 0, d, None) == -3
        assert L.rorl_gemm_nt(d, d, d, 128, 128, 256, 1, 128, 128, 128, 0, 0, 0, 1, 0, passes, None) == -3
        assert L.rorl_gemm_tn_work_bytes(128, 64, 1, 0, passes) == -3
    for N_ in (4, 260):
        assert L.rorl_gemm_tn_work_bytes(N_, 36, 1, 0, 2) == 2 * N_ * 40 * 2
        assert L.rorl_gemm_tn_work_bytes(N_, 36, 3, 4, 4) == 2 * 3 * N_ * 40 * 2
    assert L.rorl_gemm_tn_work_bytes(256, 64, 1, 0, 2) == 2 * 256 * 64 * 2
    lib = ctypes.CDLL(N.LIB_PATH)
    for name in ("rorl_gemm_force_bn", "rorl_gemm_force_bk", "rorl_gemm_debug"):
        assert not hasattr(lib, name), name


def test_kernels_refuse_cpu_tensors():
    import rorl_b200.kernels as K
    with pytest.raises(RuntimeError, match="CUDA tensors only"):
        K.real_scan_tie_input_gate(torch.zeros(1, 4, 4), torch.zeros(1, 4, 4))


def test_layer_id_grammar():
    from rorl_b200.models.rnn_base import check_is_rnn, parse_layer_id
    assert parse_layer_id('smamba_s32_c16_b2_nln') == ('smamba', dict(d_state=32, d_conv=16, block_num=2, rms_norm=False, use_ff=False))
    assert parse_layer_id('smamba_b1_c8_s64_ff')[1] == dict(d_state=64, d_conv=8, block_num=1, rms_norm=True, use_ff=True)
    assert parse_layer_id('smamba') == ('smamba', dict(d_state=16, d_conv=4, block_num=2, rms_norm=True, use_ff=False))
    assert parse_layer_id('cgpt_h8_l6_p0.1_ml1024_rms') == ('cgpt', dict(nhead=8, nlayer=6, pdrop=0.1, maxlength=1024, ln=False))
    assert parse_layer_id('efc-8') == ('efc', {'ensemble': 8})
    assert parse_layer_id('mamba_s32_c16') == ('mamba', dict(d_state=32, d_conv=16, use_ff=True))
    assert parse_layer_id('mamba_noff')[1] == dict(d_state=16, d_conv=4, use_ff=False)
    assert parse_layer_id('conv1d_8') == ('conv1d', {'d_conv': 8}) and parse_layer_id('gilr_lstm') == ('gilr_lstm', {})
    for lid in ('gru', 'lru', 'gilr', 'smamba_s16', 'cgpt_h8', 'mamba_s16', 'gilr_lstm', 'conv1d_4'):
        assert check_is_rnn(lid)
    assert not check_is_rnn('fc') and not check_is_rnn('efc-8')
    with pytest.raises(NotImplementedError):
        parse_layer_id('cgru')


@pytest.mark.parametrize("tag", ["sac_smamba", "sac_gru", "td3_gilr", "td3_lru"])
def test_state_dict_and_resel_split_compatible(tag):
    from rorl_b200.algorithm.full_length_update import prepare_param_list
    from rorl_b200.policy_value_models.make_models import make_policy_model, make_value_model
    g = load_npz(f"update_{tag}.npz")
    cfg = cfg_of(g)
    algo = cfg["case"]["algo"]
    pol = make_policy_model(cfg["policy_kwargs"], algo, False)
    val = make_value_model(cfg["value_kwargs"], algo, False)
    for model, pre in ((pol, "init/policy/"), (val, "init/value/")):
        ref = nested_sd(g, pre)
        mine = model.state_dict()
        assert list(ref) == list(mine)
        for k in ref:
            assert list(ref[k]) == list(mine[k]), k
            for n in ref[k]:
                assert tuple(ref[k][n].shape) == tuple(mine[k][n].shape), (k, n)
        model.load_state_dict(ref)
    groups = prepare_param_list(val, 1e-5, 0.0)
    slow = {id(p) for gr in groups if gr.get("lr") == 1e-5 for p in gr["params"]}
    assert slow == {id(p) for p in val.embedding_network.parameters()}
    fast = {id(p) for gr in groups if "lr" not in gr for p in gr["params"]}
    assert fast == {id(p) for k, m in val.contextual_modules.items() if k != 'embedding_model' for p in m.parameters()}
    h = val.make_init_state(3, torch.device('cpu'))
    assert len(h) == val.rnn_num and h[0].shape[:2] == (1, 3)


def _fill(buf, Transition, rng, lens, S, A):
    for Tn in lens:
        last_s, last_a, last_r = np.zeros((1, S)), np.zeros((1, A)), np.zeros((1, 1))
        s = rng.standard_normal((1, S))
        for t in range(Tn):
            a = np.tanh(rng.standard_normal((1, A)))
            ns = rng.standard_normal((1, S))
            r = float(rng.standard_normal())
            done = t == Tn - 1
            buf.mem_push(Transition(state=s, last_state=last_s, last_action=last_a, action=a, next_state=ns, reward=r,
                                    logp=None, mask=1, done=done, timeout=done, start=(t == 0), reward_input=last_r))
            last_s, last_a, last_r, s = s, a, np.array([[r]]), ns


def _apply_plan_numpy(buf, plan):
    """What csrc/gather.cu does, restated with numpy for the CPU check of the host plan."""
    F = buf.memory_buffer.shape[1]
    out = np.zeros((plan.rows, buf.max_traj_step, F))
    valid = np.zeros((plan.rows, buf.max_traj_step, 1))
    skip = buf._skip_step
    sc, mc = buf._rnn_start_range[0], buf._mask_range[0]
    for src, row, ptr, n in plan.entries:
        out[row, ptr + skip:ptr + skip + n] = buf.memory_buffer[src:src + n]
        out[row, ptr + skip - 1, buf._target_range] = buf.memory_buffer[src, buf._source_range]
        out[row, ptr:ptr + skip, sc] = 1
        valid[row, ptr + skip:ptr + skip + n, 0] = buf.memory_buffer[src:src + n, mc]
    for row, e in enumerate(plan.row_end):
        out[row, e:, sc] = 1
    out[..., mc].reshape(-1)[plan.mask_zero] = 0          # randomize_mask (a view: out is contiguous)
    return out[:, :plan.width], valid[:, :plan.width]


@pytest.mark.parametrize("tag", ["a", "b", "c", "d", "e", "f", "g", "h", "i"])
def test_sampler_plan_bit_exact(tag):
    from rorl_b200.buffers.transition_buffer.nested_replay_memory import NestedMemoryArray
    from rorl_b200.buffers.transition_buffer.replay_memory import Transition
    g = load_npz(f"sampler_{tag}.npz")
    c = cfg_of(g)
    buf = NestedMemoryArray(500, c["max_step"], additional_history_len=c["skip_extra"])
    _fill(buf, Transition, np.random.RandomState(3), c["lens"], c["S"], c["A"])
    np.random.seed(11)
    for call in range(2):
        plan = buf.plan_trajs(c["batch"], None, nest_stack_trajs=c["nest"], randomize_mask=c.get("randomize_mask", False),
                              valid_number_post_randomized=c.get("valid_num", 0),
                              equalize_data_of_each_traj=c.get("equalize", True), random_trunc_traj=c.get("random_trunc", False))
        data, valid = _apply_plan_numpy(buf, plan)
        tr = buf.array_to_transition(data)
        for n in tr._fields:
            v = getattr(tr, n)
            if v is None:
                assert f"c{call}/{n}" not in g
                continue
            assert np.array_equal(v, g[f"c{call}/{n}"]), n
        assert np.array_equal(valid, g[f"c{call}/valid"])
        assert np.array_equal(plan.lens, g[f"c{call}/lens"])
        assert plan.total_size == int(g[f"c{call}/total"])
        st = np.random.get_state()
        assert np.array_equal(np.array(st[1][:4], dtype=np.int64), g[f"c{call}/rng_next"]) and st[2] == int(g[f"c{call}/rng_pos"])
    with pytest.raises(RuntimeError, match="no CPU path"):
        buf.gather_device(plan)


def test_s6_layer_state_dict_keys_and_hidden_size():
    """s6 `mamba_*` layer: parameter names / shapes and the hidden width of the reference (layer_mamba_*.npz were
    recorded from the unmodified reference's RNNBase)."""
    from rorl_b200.models.rnn_base import RNNBase
    for tag in ("mamba_ff", "mamba_noff"):
        g = load_npz(f"layer_{tag}.npz")
        net = RNNBase(12, 8, [16, 16], ['elu', 'elu', 'linear'], ['fc', str(g["layer_id"]), 'fc'])
        ref = {k[2:]: v.shape for k, v in g.items() if k.startswith("p/")}
        mine = {k: tuple(v.shape) for k, v in net.state_dict().items()}
        assert list(ref) == list(mine)
        for k in ref:
            assert tuple(ref[k]) == mine[k], k
        assert net.rnn_hidden_state_input_size == [g["h_in"].shape[-1]]


def test_checkpoint_files_follow_reference_naming(tmp_path):
    """save()/load() write one `{name}-{index}-{module}.pt` state_dict per contextual module, the reference's
    checkpoint layout (ref: offpolicy_rnn/models/contextual_model.py:135-153)."""
    import os
    from rorl_b200.policy_value_models.make_models import make_policy_model
    kw = dict(state_dim=5, action_dim=3, embedding_size=8, embedding_hidden=[16, 16], embedding_activations=['elu', 'elu', 'linear'],
              embedding_layer_type=['fc', 'gilr', 'fc'], uni_model_hidden=[16, 16], uni_model_activations=['elu', 'elu', 'linear'],
              uni_model_layer_type=['fc'] * 3, fix_rnn_length=0, uni_model_input_mapping_dim=8, reward_input=False,
              last_action_input=True, last_state_input=True, separate_encoder=True)
    torch.manual_seed(0)
    a = make_policy_model(kw, 'sac', False)
    torch.manual_seed(1)
    b = make_policy_model(kw, 'sac', False)
    a.save(str(tmp_path), 7)
    files = sorted(os.listdir(tmp_path))
    assert files == sorted(f"{a.name}-7-{k}.pt" for k in a.contextual_modules)
    b.load(str(tmp_path), 7)
    for k, sd in a.state_dict().items():
        for n, t in sd.items():
            assert torch.equal(t, b.state_dict()[k][n]), (k, n)
