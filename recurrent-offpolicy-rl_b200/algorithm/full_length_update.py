"""The recurrent off-policy update hot path: `train_one_batch()` of the full-length-trajectory SAC / TD3
algorithms with ensemble-Q / REDQ targets and the RESeL per-encoder learning-rate split.

Mirrors, step for step, the reference's
  SACFullLengthRNNEnsembleQ.train_one_batch   ref: offpolicy_rnn/algorithm/sac_full_length_rnn_ensembleQ.py:297-467
  _target_Q / _Q_loss / _policy_loss / _alpha_loss                                   :83-132
  REDQ subset + mean aggregate                ref: sac_full_length_rnn_redq.py:16-47
  TD3 targets / actor                         ref: td3_full_length_rnn_ensembleQ.py:23-71, td3_full_length_rnn_redq.py:14-50
  prepare_param_list (RESeL groups)           ref: sac_full_length_rnn_redq_sep_optim.py:37-102
  optimizers / log_alpha / target entropy     ref: sac.py:61-95
with the B200-native restructuring:
  * the batch never visits the host: host integer plan -> device gather (buffers/...nested_replay_memory.py);
  * parameters, gradients, Adam moments and target parameters of each model live in flat fp32 arenas, so the
    AdamW step + Polyak target update is ONE kernel per model (csrc/optim.cu) and a data-parallel gradient
    all-reduce is ONE NCCL call per model;
  * target-Q / guard / masked-TD / actor / entropy reductions are fused kernels producing the loss AND the
    gradient seeds (csrc/losses.cu); no `.item()` inside the update -- logged scalars are gathered in one
    device vector and read back once (or not at all with `sync=False`);
  * the value network's parameters are frozen during the actor pass (the reference computes and then discards
    those gradients, ref :122-123,268).
"""
from __future__ import annotations

import math
import os
from types import SimpleNamespace
from typing import Dict, List, Optional

import numpy as np
import torch

from .. import _native as N
from .. import kernels as K
from ..buffers.transition_buffer.nested_replay_memory import NestedMemoryArray
from ..policy_value_models.make_models import make_policy_model, make_value_model
from ..utility.q_value_guard import QValueGuard
from .data_parallel import BucketedGradSync, sync_count_and_guard

DEFAULTS = dict(utd=1, policy_utd=1, randomize_mask=False, valid_number_post_randomized=0, random_trunc_traj=False,
                randomize_first_hidden=False, gamma=0.99, sac_tau=0.995, policy_update_per=1, no_alpha_auto_tune=False,
                use_cuda_graph=True, policy_max_gradnorm=None, policy_embedding_max_gradnorm=None, value_max_gradnorm=None,
                value_embedding_max_gradnorm=None, redq_m=2, target_action_noise_std=0.04,
                target_action_noise_clip=0.12, policy_lr=3e-4, value_lr=1e-3, rnn_policy_lr=1e-5, rnn_value_lr=1e-4,
                alpha_lr=1e-2, policy_l2_norm=0.0, value_l2_norm=0.0, sample_std=0.1, target_entropy_ratio=1.5,
                sac_alpha=1.0, value_net_num=1, max_buffer_transition_num=1000000, sac_batch_size=1000)


# ------------------------------------------------------------------------------------------------------------------
# RESeL parameter groups (API-compatible helper) and the flat arena built from them
# ------------------------------------------------------------------------------------------------------------------
def prepare_param_list(model, rnn_lr, l2_norm):
    """Param groups exactly as the reference builds them: modules whose name ends with 'encoder' and everything
    that is not `embedding_model` keep the optimizer's base lr; every layer of the embedding network (pre-fc,
    RNN, post-fc, norms) gets `rnn_lr` (ref: sac_full_length_rnn_redq_sep_optim.py:49-79)."""
    groups = []
    for k, v in model.contextual_modules.items():
        kind = type(v).__name__
        if k == 'embedding_model':
            mods = [v.layer_list[0]] + [v.layer_list[i] for i in range(1, len(model.embedding_network.layer_list) - 1)] \
                   + [v.layer_list[-1], v.activation_list]
            for m in mods:
                groups.append({"params": list(m.parameters(True)), "lr": rnn_lr, "weight_decay": l2_norm, "name": f"rnn-{kind}"})
        else:
            groups.append({"params": list(v.parameters(True)), "name": f"mlp-{kind}"})
    return groups


class FlatArena:
    """All parameters of one model re-homed as views of one flat fp32 buffer (plus flat grad / Adam moments)."""

    def __init__(self, model, device, grad_tail: int = 0):
        """`grad_tail` extra floats at the end of the gradient buffer (not of the parameters): a slot that rides along
        in the arena's data-parallel all-reduce (the policy arena carries the log-alpha gradient there)."""
        params = [p for p in model.parameters(True)]
        seen, uniq = set(), []
        for p in params:
            if id(p) not in seen:
                seen.add(id(p))
                uniq.append(p)
        self.params = uniq
        self.offsets, n = [], 0
        for p in uniq:
            self.offsets.append(n)
            n += (p.numel() + 3) // 4 * 4          # keep every tensor 16-byte aligned inside the arena
        self.numel = n
        self.flat = torch.zeros(n, dtype=torch.float32, device=device)
        self.grad_full = torch.zeros(n + grad_tail, dtype=torch.float32, device=device)
        self.grad = self.grad_full[:n]
        self.tail = self.grad_full[n:]
        with torch.no_grad():
            for p, off in zip(uniq, self.offsets):
                self.flat[off:off + p.numel()].copy_(p.data.reshape(-1))
                p.data = self.flat[off:off + p.numel()].view(p.shape)
                p.grad = self.grad[off:off + p.numel()].view(p.shape)

    def offset_of(self, p) -> int:
        for q, off in zip(self.params, self.offsets):
            if q is p:
                return off
        raise KeyError

    def _views(self):
        if getattr(self, '_view_cache', None) is None:
            self._view_cache = [self.grad[off:off + p.numel()].view(p.shape) for p, off in zip(self.params, self.offsets)]
        return self._view_cache

    def zero_grad(self, detach: bool = False):
        """detach=False: `.grad` stays the arena view and autograd accumulates into it (one add_ launch per parameter; what
        the bucketed data-parallel hooks need).  detach=True: `.grad` is dropped so that autograd keeps each produced
        gradient by reference, and `collect()` moves them all into the arena with one multi-tensor copy."""
        self.grad_full.zero_()
        if detach:
            for p in self.params:
                p.grad = None
            return
        for p, v in zip(self.params, self._views()):      # autograd may have swapped .grad out; put the view back
            if p.grad is None or p.grad.data_ptr() != v.data_ptr():
                p.grad = v

    def collect(self):
        """After a backward run with zero_grad(detach=True): gather the gradients into the (zeroed) arena, re-point `.grad`."""
        srcs, dsts = [], []
        for p, v in zip(self.params, self._views()):
            g = p.grad
            if g is not None and g.data_ptr() != v.data_ptr():
                srcs.append(g if g.shape == v.shape else g.reshape(v.shape))
                dsts.append(v)
            p.grad = v
        if srcs:
            torch._foreach_copy_(dsts, srcs)


class FusedAdamW:
    """AdamW(betas=(0.9, 0.999), eps=1e-8) over a FlatArena with contiguous lr / weight-decay / clip-value segments,
    fused with the Polyak target update when a target arena is given, and with the reference's gradient clipping
    (csrc/optim.cu): `max_norm` = clip_grad_norm_ over the whole model, `clip_values` = {id(param): bound} for
    clip_grad_value_ (ref: sac_full_length_rnn_ensembleQ.py:239-250,274-287)."""

    def __init__(self, arena: FlatArena, groups: List[dict], lr: float, weight_decay: float, target: Optional[FlatArena] = None,
                 max_norm: Optional[float] = None, clip_values: Optional[Dict[int, float]] = None, work: Optional[torch.Tensor] = None,
                 gnorm_out: Optional[torch.Tensor] = None):
        self.arena, self.target = arena, target
        dev = arena.flat.device
        self.m = torch.zeros_like(arena.flat)
        self.v = torch.zeros_like(arena.flat)
        self.step_count = torch.zeros(1, dtype=torch.int32, device=dev)
        self.max_norm = None if max_norm is None else float(max_norm)
        self.gnorm_sq = gnorm_out if gnorm_out is not None else torch.zeros(1, dtype=torch.float32, device=dev)
        self._work = work
        self._per_param = {}
        for g in groups:
            for p in g["params"]:
                self._per_param[id(p)] = (g.get("lr", lr), g.get("weight_decay", weight_decay))
        self._clip_values = dict(clip_values or {})
        self._frozen = set()
        self._build_segments()

    def _build_segments(self):
        dev = self.arena.flat.device
        ends, cfgs = [], []
        for p, off in zip(self.arena.params, self.arena.offsets):
            lr_, wd_ = self._per_param[id(p)]
            if id(p) in self._frozen:            # torch.optim skips parameters whose .grad is None: no step, no decay
                lr_, wd_ = 0.0, 0.0
            cfg = (lr_, wd_, float(self._clip_values.get(id(p), 0.0)))
            end = off + (p.numel() + 3) // 4 * 4
            if cfgs and cfgs[-1] == cfg:
                ends[-1] = end
            else:
                ends.append(end), cfgs.append(cfg)
        assert len(ends) <= 64, 'too many lr segments; order modules so that groups are contiguous'
        self.param_groups = [{"lr": c[0], "weight_decay": c[1], "clip_value": c[2], "end": e} for c, e in zip(cfgs, ends)]
        self.seg_end = torch.tensor(ends, dtype=torch.int64, device=dev)
        self.seg_lr = torch.tensor([c[0] for c in cfgs], dtype=torch.float64, device=dev)
        self.seg_wd = torch.tensor([c[1] for c in cfgs], dtype=torch.float64, device=dev)
        self.seg_clip = torch.tensor([c[2] for c in cfgs], dtype=torch.float64, device=dev) if any(c[2] > 0 for c in cfgs) else None

    def freeze_params_without_grad(self, got_grad: Dict[int, bool]):
        """Parameters that never receive a gradient (e.g. GILRLayer.layer_norm, constructed but unused) keep
        `.grad is None` in the reference, so torch.optim.AdamW skips them -- no weight decay either."""
        frozen = {id(p) for p in self.arena.params if not got_grad.get(id(p), False)}
        if frozen != self._frozen:
            self._frozen = frozen
            self._build_segments()
            return True
        return False

    def zero_grad(self, detach: bool = False):
        self.arena.zero_grad(detach)

    def step(self, tau: Optional[float] = None):
        tgt = self.target.flat if (self.target is not None and tau is not None) else None
        gn = None
        if self.max_norm is not None:
            N.call("rorl_sumsq", N.ptr(self.arena.grad), self.arena.numel, N.ptr(self.gnorm_sq), N.ptr(self._work), N.stream())
            gn = self.gnorm_sq
        N.call("rorl_adamw_polyak", N.ptr(self.arena.flat), N.ptr(self.arena.grad), N.ptr(self.m), N.ptr(self.v),
               N.ptr(tgt), N.ptr(self.seg_end), N.ptr(self.seg_lr), N.ptr(self.seg_wd), N.ptr(self.seg_clip),
               len(self.param_groups), self.arena.numel, 0.9, 0.999, 1e-8, float(tau if tau is not None else 1.0),
               N.ptr(self.step_count), N.ptr(gn), float(self.max_norm or 0.0), N.stream())


# ------------------------------------------------------------------------------------------------------------------
# the update
# ------------------------------------------------------------------------------------------------------------------
class FullLengthRNNUpdate:
    """Holds what `train_one_batch` of the reference algorithm object touches (SURVEY.md App. D) and runs it.

    Environment construction, rollout, evaluation and logging (ref: algorithm/sac.py:34-127,274-401) are out of
    scope, so instead of reading them from an env the constructor takes `obs_dim`, `act_dim`,
    `max_trajectory_len` and the model kwargs the reference derives from its flags (ref: sac.py:199-239).
    """
    base_algorithm = 'sac'
    use_redq = True
    sep_optim = False           # RESeL per-encoder learning-rate split: only the *_SEP_OPTIM classes (ref: sac.py:81-90 otherwise)

    def __init__(self, parameter, policy_args: dict, value_args: dict, max_trajectory_len: int, device=None,
                 dist_group=None, discrete_env: bool = False):
        hp = dict(DEFAULTS)
        hp.update(parameter if isinstance(parameter, dict) else vars(parameter))
        self.parameter = SimpleNamespace(**hp)
        if device is None:
            device = torch.device('cuda', torch.cuda.current_device())
        self.device = self.sample_device = torch.device(device)
        if self.device.type != 'cuda':
            raise RuntimeError('the update hot path runs on sm_100a kernels only; no CPU path exists')
        self.discrete_env = bool(discrete_env)
        self.dist_group = dist_group
        td3 = self.base_algorithm == 'td3'
        if self.discrete_env:
            # ref: sac.py:72-74 (discrete action space: fixed alpha), sac_full_length_rnn_ensembleQ.py:43-44 (guard decay 1)
            assert not td3, 'the TD3 classes have no discrete-action variant in the reference'
            self.parameter.no_alpha_auto_tune = True
        if td3:
            self.parameter.no_alpha_auto_tune = True
            policy_args = dict(policy_args, sample_std=self.parameter.sample_std)
        self.policy_args, self.value_args = policy_args, value_args
        assert self.parameter.value_net_num == 1
        for item in value_args['uni_model_layer_type']:
            assert item.startswith('e')
        # models (ref: sac.py:61-70) --------------------------------------------------------------------------
        self.policy = make_policy_model(policy_args, self.base_algorithm, self.discrete_env)
        self.values = [make_value_model(value_args, self.base_algorithm, self.discrete_env)]
        self.target_values = [make_value_model(value_args, self.base_algorithm, self.discrete_env)]
        self.target_policy = make_policy_model(policy_args, self.base_algorithm, self.discrete_env)
        for m in [self.policy, self.target_policy] + self.values + self.target_values:
            m.to(self.device)
        for net in (self.values[0].embedding_network.layer_list + self.target_values[0].embedding_network.layer_list
                    + self.values[0].uni_network.layer_list + self.target_values[0].uni_network.layer_list):
            if hasattr(net, 'desire_ndim'):                      # ref: sac_full_length_rnn_ensembleQ.py:25-32
                net.desire_ndim = 4
            if hasattr(net, 'in_proj') and hasattr(net.in_proj, 'desire_ndim'):
                net.in_proj.desire_ndim = 4
        a0 = math.log(self.parameter.sac_alpha) if self.parameter.no_alpha_auto_tune else 0.0
        self.log_sac_alpha = torch.tensor([a0], dtype=torch.float32, device=self.device, requires_grad=True)
        self.target_entropy = (self.parameter.target_entropy_ratio if self.discrete_env            # ref: sac.py:80
                               else -float(policy_args['action_dim']) * self.parameter.target_entropy_ratio)
        self.replay_buffer = NestedMemoryArray(self.parameter.max_buffer_transition_num, max_trajectory_len,
                                               additional_history_len=self._get_skip_len(), device=self.device)
        self.Q_guard = QValueGuard(True, True, 1.0 if self.discrete_env else 1 - 1e-3, device=self.device)
        self.allow_nest_stack = self.allow_nest_stack_trajs()
        self.grad_num = 0
        # scratch for the fused reductions
        self._work = torch.zeros(int(N.lib().rorl_loss_work_floats(0)), dtype=torch.float32, device=self.device)
        self._stats = torch.zeros(16, dtype=torch.float32, device=self.device)
        self._finalize_models()
        self._ensemble_size = int(value_args['uni_model_layer_type'][-1].split('-')[-1])
        self._h2d_stage = None
        self._has_gpt = any('gpt' in lid for net in (self.values[0].embedding_network, self.policy.embedding_network,
                                                     self.values[0].uni_network, self.policy.uni_network) for lid in net.layer_type)
        env = os.environ.get('RORL_CUDA_GRAPH')
        self.use_cuda_graph = bool(hp.get('use_cuda_graph', True)) if env is None else env not in ('0', 'false', 'off')
        self._graphs: Dict = {}
        self._graph_pool = None

    # ---- construction helpers ---------------------------------------------------------------------------------
    def _finalize_models(self):
        """(Re)build arenas + optimizers after weights are in place; call again after load_state_dict."""
        self._graphs, self._graph_pool = {}, None       # captured graphs point into the old arenas
        for m in [self.policy, self.target_policy] + list(self.values) + list(self.target_values):
            m.need_full_hidden = False                  # the update never reads forward()'s per-layer output record
        gpt = any(str(t).startswith(('cgpt', 'gpt', 'transformer')) for m in (self.policy, self.values[0])
                  for t in m.embedding_network.layer_type)
        side_ok = (self.device.type == 'cuda' and not gpt       # cgpt: device-side dropout counter order
                   and os.environ.get('RORL_SIDE_STREAM', '1') != '0')
        self._side_stream = torch.cuda.Stream(device=self.device) if side_ok else None
        self._has_gru = any(str(t) == 'gru' for m in (self.policy, self.values[0]) for t in m.embedding_network.layer_type)
        self._value_update(tau=0.0)
        self.target_policy.copy_weight_from(self.policy, tau=0.0)
        self.policy_arena = FlatArena(self.policy, self.device, grad_tail=4)
        self.value_arena = FlatArena(self.values[0], self.device)
        self.target_arena = FlatArena(self.target_values[0], self.device)
        # the log-alpha gradient lives in the tail slot of the policy gradient arena: one all-reduce carries both
        self.alpha_arena = SimpleNamespace(flat=self.log_sac_alpha.data, grad=self.policy_arena.tail[:1],
                                           params=[self.log_sac_alpha], offsets=[0], numel=1, zero_grad=lambda: None)
        self._guard_init_synced = False
        # bf16 hi | lo copies of the weights as the GEMMs' B operands, kept across the ~110 GEMM calls of an update and rebuilt
        # by one launch per arena whenever that arena changes (kernels.WeightSplitCache)
        self._split_cache = None
        if self.device.type == 'cuda' and os.environ.get('RORL_SPLIT_CACHE', '1') != '0':
            self._split_cache = K.WeightSplitCache(self.device)
            self._split_owner = {name: self._split_cache.add_owner(a.flat) for name, a in
                                 (('policy', self.policy_arena), ('value', self.value_arena), ('target', self.target_arena))}
        p = self.parameter

        def groups(model, rnn_lr, l2):
            # RESeL groups only in the *_SEP_OPTIM classes; otherwise one AdamW over all parameters (ref: sac.py:81-90)
            return prepare_param_list(model, rnn_lr, l2) if self.sep_optim else [{"params": list(model.parameters(True))}]

        def clip_values(model, bound):
            """clip_grad_value_ on the embedding network, then the hard-coded 1e-3 on every smamba A_log
            (ref: sac_full_length_rnn_ensembleQ.py:244-250,279-287)."""
            if bound is None:
                return None
            out = {id(q): float(bound) for q in model.embedding_network.parameters(True)}
            for layer in model.embedding_network.layer_list:
                for sub in getattr(layer, 'layers', []):
                    a_log = getattr(getattr(sub, 'mixer', None), 'A_log', None)
                    if a_log is None:
                        break                       # the reference's try/except leaves the layer at the first miss
                    out[id(a_log)] = min(float(bound), 1e-3)
            return out

        self.optimizer_policy = FusedAdamW(self.policy_arena, groups(self.policy, p.rnn_policy_lr, p.policy_l2_norm),
                                           p.policy_lr, p.policy_l2_norm, max_norm=p.policy_max_gradnorm,
                                           clip_values=clip_values(self.policy, p.policy_embedding_max_gradnorm), work=self._work,
                                           gnorm_out=self._stats[11:12])
        self.optimizer_value = FusedAdamW(self.value_arena, groups(self.values[0], p.rnn_value_lr, p.value_l2_norm),
                                          p.value_lr, p.value_l2_norm, target=self.target_arena, max_norm=p.value_max_gradnorm,
                                          clip_values=clip_values(self.values[0], p.value_embedding_max_gradnorm), work=self._work,
                                          gnorm_out=self._stats[10:11])
        # torch.optim.AdamW's default weight_decay (1e-2) applies: the reference passes only lr (ref: sac.py:90)
        self.optimizer_alpha = FusedAdamW(self.alpha_arena, [{"params": [self.log_sac_alpha]}], p.alpha_lr, 1e-2)
        self._grad_seen = None                         # first update: learn which parameters ever receive a gradient
        for h in (getattr(self, '_grad_hooks', None) or []):
            h.remove()
        self._grad_hooks = None
        self._opt_steps = {'value': 0, 'policy': 0}    # completed optimizer steps (GradScaler growth emulation, see _amp_scale)
        # l2_norm_square() covers the RNNBase modules only (ref: contextual_model.py:227-228): a prefix of each arena
        self._l2_span = {}
        for name, model, arena in (('policy', self.policy, self.policy_arena), ('value', self.values[0], self.value_arena)):
            ids = {id(q) for m in model.contextual_modules.values() if hasattr(m, 'l2_norm_square') for q in m.parameters(True)}
            flags = [id(q) in ids for q in arena.params]
            n_in = sum(flags)
            assert all(flags[:n_in]) and not any(flags[n_in:]), 'RNNBase modules must lead the arena'
            self._l2_span[name] = arena.offsets[n_in] if n_in < len(arena.params) else arena.numel
        self.value_parameters = list(self.values[0].parameters(True))
        for m in self.values:
            m.train()
        for m in self.target_values:
            m.eval()
        self.target_policy.eval()
        self.policy.train()
        for q in self.target_arena.params + list(self.target_policy.parameters(True)):
            q.requires_grad_(False)
        # data parallel: bucketed gradient all-reduce overlapped with the backward pass (algorithm/data_parallel.py)
        for old in (getattr(self, '_sync_value', None), getattr(self, '_sync_policy', None)):
            if old is not None:
                old.remove()
        self._sync_value = self._sync_policy = None
        if self.dist_group is not None:
            self._sync_value = BucketedGradSync(self.value_arena.params, self.value_arena.offsets, self.value_arena.grad, self.dist_group)
            self._sync_policy = BucketedGradSync(self.policy_arena.params, self.policy_arena.offsets, self.policy_arena.grad, self.dist_group)

    def invalidate_graphs(self):
        """Drop every captured CUDA graph.  Scalars that are plain Python numbers at launch time (gamma, tau, the
        target entropy, noise scales) are baked into a captured graph, so call this after changing a hyper-parameter
        on a live object; weights, optimizer state and learning-rate tables live in device memory and need no
        re-capture.  (`load_models` / `_finalize_models` call it themselves: the arenas move.)"""
        self._graphs, self._graph_pool = {}, None

    def load_models(self, policy_sd=None, value_sd=None):
        if policy_sd is not None:
            self.policy.load_state_dict(policy_sd)
        if value_sd is not None:
            self.values[0].load_state_dict(value_sd)
        self._finalize_models()

    def _get_skip_len(self):
        """1 + widest causal-conv window of any encoder layer (ref: sac_full_length_rnn_ensembleQ.py:57-68)."""
        skip = 0
        for net in (self.values[0].uni_network, self.values[0].embedding_network, self.policy.uni_network,
                    self.policy.embedding_network):
            for lid, layer in zip(net.layer_type, net.layer_list):
                if 'smamba' in lid:
                    skip = max(skip, layer.d_conv)
                elif 'mamba' in lid:
                    skip = max(skip, layer.mixer.d_conv)
                elif 'conv1d' in lid:
                    skip = max(skip, layer.d_conv)
        return skip + 1

    def allow_nest_stack_trajs(self):
        """ref: sac.py:130-138"""
        for net in (self.values[0].uni_network, self.values[0].embedding_network, self.policy.uni_network,
                    self.policy.embedding_network):
            for lid in net.layer_type:
                if 'transformer' in lid or 'gru' in lid:
                    return False
        return True

    def _value_update(self, tau):
        for v, t in zip(self.values, self.target_values):
            t.copy_weight_from(v, tau)

    # ---- fused reductions -----------------------------------------------------------------------------------------
    def _target_Q(self, q_next, sel_idx, logp_next, reward, done, timeout, mask):
        """y = r + (1 - done') * gamma * clamp(min_{sel} Q' - alpha * logp') and the guard update; fills
        stats[0] = max|y|, stats[1] = n_valid."""
        E, M = q_next.shape[0], q_next[0].numel()
        m = torch.empty(M, dtype=torch.float32, device=self.device)
        sel = sel_idx                                                  # int32 device tensor [m]
        # every operand is bound to a local until its launch is enqueued: a temporary freed right after
        # data_ptr() would hand its block to the next temporary and the pointers would alias.
        qn = q_next.contiguous()
        lp = None if logp_next is None else logp_next.contiguous()
        N.call("rorl_target_minq", N.ptr(qn), N.ptr(sel), int(sel.numel()), E, M, N.ptr(lp), N.ptr(self.log_sac_alpha.data),
               N.ptr(m), N.ptr(self.Q_guard.state), N.ptr(self._work), N.stream())
        return self._target_finish(m, reward, done, timeout, mask)

    def _target_finish(self, m, reward, done, timeout, mask):
        """y = r + (1 - done') * gamma * clamp(m) and the guard update, from the per-step value m [M] whose kernel has
        initialised the guard on its first call; fills stats[0] = max|y|, stats[1] = n_valid."""
        M = m.numel()
        r_c, d_c, t_c, m_c = reward.contiguous(), done.contiguous(), timeout.contiguous(), mask.contiguous()
        y = torch.empty_like(r_c)
        if self.dist_group is not None and not self._guard_init_synced:
            # very first call (always launched eagerly): the guard bounds were just initialised from THIS rank's rows;
            # make them the global extrema before the clamp / update uses them (ref: q_value_guard.py:22-27)
            import torch.distributed as dist
            dist.all_reduce(self.Q_guard.state[0:1], op=dist.ReduceOp.MIN, group=self.dist_group)
            dist.all_reduce(self.Q_guard.state[1:2], op=dist.ReduceOp.MAX, group=self.dist_group)
            self._guard_init_synced = True
        N.call("rorl_target_finish", N.ptr(m), N.ptr(r_c), N.ptr(d_c), N.ptr(t_c), N.ptr(m_c), float(self.parameter.gamma),
               N.ptr(y), N.ptr(self.Q_guard.state), N.ptr(self._stats), N.ptr(self._work), M, N.stream())
        return y

    def _allreduce(self, t, op=None):
        if self.dist_group is not None:
            import torch.distributed as dist
            dist.all_reduce(t, op=op or dist.ReduceOp.SUM, group=self.dist_group)

    # ---- the hot path -----------------------------------------------------------------------------------------------
    def train_one_batch(self, sync: bool = True) -> Dict:
        """Sample trajectory batches from the device-resident replay and run `utd` updates on them (ref :311-434):
        every iteration updates the critic; the actor / alpha follow the reference's cadence
        `grad_num % policy_update_per == 0 and (utd_idx + 1) / utd * policy_utd > policy_update_cnt` (ref :405)."""
        p = self.parameter
        out, policy_update_cnt = None, 0
        for utd_idx in range(p.utd):
            # 1. sample (host plan, device gather) --------------------------------------------------- ref :313-332
            batch, batch_size, valid_ind, traj_len_array = self.replay_buffer.sample_trajs_device(
                p.sac_batch_size, None, randomize_mask=p.randomize_mask, valid_number_post_randomized=p.valid_number_post_randomized,
                equalize_data_of_each_traj=True, random_trunc_traj=p.random_trunc_traj, nest_stack_trajs=self.allow_nest_stack)
            did_policy = (self.grad_num % p.policy_update_per == 0) and ((utd_idx + 1) / p.utd * p.policy_utd > policy_update_cnt)
            out = self.update_on_batch(batch, batch_size, valid_ind, traj_len_array, sync=sync and utd_idx == p.utd - 1,
                                       did_policy=did_policy, advance=False, policy_logged=policy_update_cnt > 0)
            policy_update_cnt += int(did_policy)
        self.grad_num += 1                                  # the caller's `grad_num += 1` (ref: sac.py:359-362)
        return out

    def update_on_host_batch(self, host_batch: torch.Tensor, host_valid: torch.Tensor, batch_size: int,
                             traj_len_array: np.ndarray, sync: bool = True) -> Dict:
        """End-to-end entry for callers that sample on the host, as the reference does (ref :313-332): the
        [rows, W, F] fp32 batch and [rows, W, 1] valid indicator come from (pinned) host memory."""
        stage = self._h2d_stage
        if stage is None or stage[0].shape != host_batch.shape or stage[1].shape != host_valid.shape:
            stage = self._h2d_stage = (torch.empty(host_batch.shape, dtype=torch.float32, device=self.device),
                                       torch.empty(host_valid.shape, dtype=torch.float32, device=self.device))
        batch, valid = stage                         # persistent device staging: same addresses every step (graph replay)
        batch.copy_(host_batch, non_blocking=True)
        valid.copy_(host_valid, non_blocking=True)
        return self.update_on_batch(self.replay_buffer.array_to_transition(batch), batch_size, valid, traj_len_array, sync=sync)

    def update_on_batch(self, batch, batch_size, valid_ind, traj_len_array, sync: bool = True, did_policy: Optional[bool] = None,
                        advance: bool = True, policy_logged: bool = False) -> Dict:
        """One update on a device-resident batch.  Host side: the REDQ subset draw (numpy global RNG, same call
        order as the reference: after the sampler's draws, ref :313 then sac_full_length_rnn_redq.py:28), the
        attention length tables, the policy-update cadence.  Device side: the segments of `_stages`, either launched eagerly
        or -- when the batch lives in persistent buffers and nothing host-dependent is baked into the launch
        sequence -- replayed from a CUDA graph captured on the second sighting of the same (buffers, shape,
        length table, cadence) key."""
        p = self.parameter
        dev = self.device
        B, L = batch.state.shape[0], batch.state.shape[1]
        E = self._ensemble_size
        sel_np = np.random.permutation(E)[:p.redq_m] if self.use_redq else np.arange(E)
        if did_policy is None:
            did_policy = self.grad_num % p.policy_update_per == 0 and p.policy_utd > 0
        # a fresh pinned staging tensor per step: the host runs ahead of the stream, and the caching host allocator does
        # not hand the block out again before the asynchronous copy that reads it has completed
        sel_pinned = torch.from_numpy(np.asarray(sel_np, dtype=np.int32)).pin_memory()
        att_np = np.zeros((B, L), dtype=np.int32)                                                      # ref :358-366
        k = min(traj_len_array.shape[1], L)
        att_np[:, :k] = traj_len_array[:, :k].astype(np.int32)
        tgt_np = np.concatenate((att_np[:, 1:], np.zeros((B, 1), dtype=np.int32)), axis=-1)
        key = None
        if self._graph_allowed():
            key = (batch.state.data_ptr(), valid_ind.data_ptr(), B, L, tuple(batch.state.stride()), did_policy,
                   len(sel_np), att_np.tobytes())
        entry = self._graphs.get(key) if key is not None else None
        if entry is not None and entry != 'seen':
            entry['sel'].copy_(sel_pinned, non_blocking=True)
            for graph, comm in entry['segments']:
                graph.replay()
                if comm is not None:
                    comm()                                  # data-parallel exchange: eager NCCL between replayed segments
            N.add_launches(entry['launches'])
        else:
            sel = torch.empty(len(sel_np), dtype=torch.int32, device=dev)
            sel.copy_(sel_pinned, non_blocking=True)
            att = torch.from_numpy(att_np).pin_memory().to(dev, non_blocking=True)
            tgt_att = torch.from_numpy(tgt_np).pin_memory().to(dev, non_blocking=True)
            att._host, tgt_att._host = att_np, tgt_np      # host copy for the cgpt work list (no device->host sync)
            ctx = {'batch': batch, 'valid_ind': valid_ind, 'att': att, 'tgt_att': tgt_att, 'sel': sel, 'did_policy': did_policy}
            if entry == 'seen':
                # second sighting: capture each segment (nothing executes during capture) and replay it at once, so
                # that the next segment is captured against the state this one leaves; the data-parallel exchanges
                # run eagerly between the segments (NCCL is kept out of the graphs)
                torch.cuda.synchronize(dev)
                l0 = N.launch_count()
                segments = []
                for stage, comm in self._stages(graph_mode=True):
                    graph = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(graph, pool=self._graph_pool, capture_error_mode="thread_local"), self._splits_active():
                        stage(ctx)
                    if self._graph_pool is None:
                        self._graph_pool = graph.pool()
                    graph.replay()
                    if comm is not None:
                        comm()
                    segments.append((graph, comm))
                self._graphs[key] = {'segments': segments, 'sel': sel, 'launches': N.launch_count() - l0, 'keep': ctx}
            else:
                if key is not None:
                    if len(self._graphs) >= 8:                          # bounded: drop the oldest key
                        self._graphs.pop(next(iter(self._graphs)))
                    self._graphs[key] = 'seen'
                self._arm_grad_detection()
                for stage, comm in self._stages(graph_mode=False):
                    with self._splits_active():
                        stage(ctx)
                    if comm is not None:
                        comm()
                if self._split_cache is not None:
                    self._split_cache.prepare()             # job tables of the operands first seen in this call (outside capture)
        if advance:
            self.grad_num += 1
        self._opt_steps['value'] += 1
        self._opt_steps['policy'] += int(did_policy)
        # logged scalars: one device vector, one read-back ------------------------------------------------------ ref :435-467
        out = {'real_batch_size': batch_size, 'real_batch_traj_num': B, 'policy_updated': did_policy}
        if not sync:
            out['stats_device'] = self._stats
            return out
        stats = self._stats
        if self.dist_group is not None:          # per-rank partial sums (already divided by the global n_valid) -> global
            import torch.distributed as dist
            stats = self._stats.clone()
            dist.all_reduce(stats[2:8], op=dist.ReduceOp.SUM, group=self.dist_group)
            dist.all_reduce(stats[0:1], op=dist.ReduceOp.MAX, group=self.dist_group)
        s = stats.tolist()
        g = self.Q_guard.state.tolist()
        clipping_emb_v = p.value_embedding_max_gradnorm is not None
        out.update({'critic_loss': s[2], 'target_q_max': s[0], 'log_alpha': float(self.log_sac_alpha.item()),
                    'clip_min': g[0], 'clip_max': g[1],
                    'value_grad_norm': (math.sqrt(s[10]) if (p.value_max_gradnorm is not None and not clipping_emb_v) else 0.0),
                    'q1_l2_norm_square': s[8],
                    'average_traj_len': self.replay_buffer.size / max(len(self.replay_buffer), 1),
                    'amp_scalar_pi': self._amp_scale('policy'), 'amp_scalar_q': self._amp_scale('value')})
        if did_policy or policy_logged:
            clipping_emb_p = p.policy_embedding_max_gradnorm is not None
            out.update({'actor_loss': s[4], 'log_prob': s[5], 'policy_l2_norm_square': s[9],
                        'policy_grad_norm': (math.sqrt(s[11]) if (p.policy_max_gradnorm is not None and not clipping_emb_p) else 0)})
            if not p.no_alpha_auto_tune:
                out['alpha_loss'] = s[6]
        return out

    def _amp_scale(self, which: str) -> float:
        """The reference wraps both optimizers in a GradScaler when any `gpt` layer is present (ref :34-40,234-258) and
        logs its scale.  Its autocast region is bf16, whose exponent range is fp32's: scaling the loss by a power of two
        and un-scaling the gradients is exact and never overflows where fp32 would not, so no scaling is applied here;
        the logged value follows GradScaler's schedule (65536, doubled every 2000 un-skipped steps)."""
        if not self._has_gpt:
            return 0
        return 65536.0 * 2.0 ** (self._opt_steps[which] // 2000)

    def _splits_active(self):
        import contextlib
        return self._split_cache.active() if self._split_cache is not None else contextlib.nullcontext()

    def _splits(self, refresh=(), invalidate=()):
        if self._split_cache is None:
            return
        for name in refresh:
            self._split_cache.refresh(self._split_owner[name])
        for name in invalidate:
            self._split_cache.invalidate(self._split_owner[name])

    def _beside(self, fn):
        """Launch fn() -- a no-grad forward that the caller's next launches do not depend on -- on the side stream, so that
        it runs BESIDE them; returns a join() that makes the current stream wait for it and hands back fn's result.
        Used for the two places where the update runs two independent context encoders back to back (target policy ||
        target value; actor's policy || the critic's encoder under the actor): a 0.86-wave scan grid, a 4-SM GRU
        recurrence or a short elementwise kernel leaves SMs idle that the other encoder's kernels can use.
        Works unchanged under CUDA-graph capture (fork / join through events on the capture stream).  No
        record_stream is needed: the results are consumed on the current stream before the next fork, and every fork
        starts by making the side stream wait for the current one."""
        if self._side_stream is None:
            res = fn()
            return lambda: res
        cur = torch.cuda.current_stream(self.device)
        self._side_stream.wait_stream(cur)
        if self._has_gru:                          # two recurrences at a time: each takes half the SMs (csrc/gru.cu)
            N.lib().rorl_gru_set_fwd_sms(72)
        with torch.cuda.stream(self._side_stream), torch.no_grad():
            res = fn()
        def join():
            cur.wait_stream(self._side_stream)
            if self._has_gru:
                N.lib().rorl_gru_set_fwd_sms(148)
            return res
        return join

    def _graph_allowed(self) -> bool:
        """CUDA-graph replay needs a launch sequence that depends on nothing the host decides per step: an injected
        `noise_fn` / `sample_fn` (parity tests) returns a different tensor per call.  (The cgpt encoder's attention work list depends
        on the length table only, which is part of the graph key; it is cached on the device by the first, eager, call.)"""
        if not self.use_cuda_graph:
            return False
        if self.discrete_env:      # the categorical head's default draw (sample_fn None) is an in-kernel torch.rand draw
            return all(m.sample_fn is None or getattr(m.sample_fn, 'graph_safe', False) for m in (self.policy, self.target_policy))
        ok = lambda fn: fn is torch.randn_like or getattr(fn, 'graph_safe', False)   # device-only, same launches every call
        return all(ok(getattr(m, 'noise_fn', torch.randn_like)) for m in (self.policy, self.target_policy))

    def _stages(self, graph_mode: bool):
        """The update as (device segment, data-parallel exchange after it) pairs.  Segments only launch (no host reads,
        no pageable copies), so each can be captured into a CUDA graph; the exchanges are NCCL calls on the same
        stream.  Eager mode keeps the bucketed all-reduce overlapped with the backward pass (hooks inside the
        segment); graph mode reduces each flat gradient arena with ONE all-reduce between two replayed segments
        (a few hundred microseconds over NVLink against a 17 ms update) and keeps NCCL out of the captured graphs."""
        dist = self.dist_group is not None
        overlap = dist and not graph_mode

        def s_target(c):
            self._stage_target(c)

        def s_critic(c):
            self._stage_critic(c, overlap)

        def s_actor(c):
            self._stage_value_step_and_actor(c, overlap)

        def s_policy_step(c):
            self._stage_policy_step(c)

        def x_count():
            self._sync_guard_and_count()

        def x_value():
            self._allreduce(self.value_arena.grad)

        def x_policy():
            self._allreduce(self.policy_arena.grad_full)      # policy gradients + the log-alpha gradient in the tail slot

        return [(s_target, x_count if dist else None),
                (s_critic, x_value if (dist and not overlap) else None),
                (s_actor, x_policy if (dist and not overlap) else None),
                (s_policy_step, None)]

    def _stage_target(self, c):
        p = self.parameter
        td3 = self.base_algorithm == 'td3'
        dev = self.device
        batch, valid_ind, att, tgt_att, sel = c['batch'], c['valid_ind'], c['att'], c['tgt_att'], c['sel']
        state, action, next_state = batch.state, batch.action, batch.next_state
        done, mask, reward, timeout, rnn_start = batch.done, batch.mask, batch.reward, batch.timeout, batch.start
        B = state.shape[0]
        self._splits(refresh=('policy', 'value', 'target'))     # weights may have changed since the last update (steps, loads)
        # the side-band flags are read by every recurrent / conv layer of four forward passes: hand them over contiguous and
        # in fp32 ONCE here (batch.start is a column slice of the sampled batch; each kernel wrapper would otherwise copy it)
        rnn_start = rnn_start.float().contiguous()
        valid_ind = valid_ind.float().contiguous()
        # 2. target-pass side-band ------------------------------------------------------------------------ ref :338-341
        d_valid = valid_ind[:, 1:] - valid_ind[:, :-1]
        total_valid = valid_ind.clone()
        total_valid[:, :-1] = torch.where(d_valid == 1, torch.ones_like(d_valid), total_valid[:, :-1])
        d_start = rnn_start[:, 1:] - rnn_start[:, :-1]
        total_start = rnn_start.clone()
        total_start[:, :-1] = torch.where(d_start == -1, torch.zeros_like(d_start), total_start[:, :-1])
        if p.randomize_first_hidden:                          # ref :345-351: random carried state, shared by both policy passes
            mk = lambda model: model.make_rnd_init_state(B, device=dev)
            c['policy_hidden'] = target_policy_hidden = mk(self.policy)
        else:
            mk = lambda model: model.make_init_state(B, device=dev)
            c['policy_hidden'], target_policy_hidden = mk(self.policy), mk(self.policy)
        target_hidden, c['value_hidden'] = mk(self.target_values[0]), mk(self.values[0])
        for h in (target_policy_hidden, target_hidden):
            h.set_rnn_start(total_start), h.set_mask(total_valid), h.set_attention_concat_mask(tgt_att)
        c['value_hidden'].set_rnn_start(rnn_start), c['value_hidden'].set_mask(valid_ind), c['value_hidden'].set_attention_concat_mask(att)
        c['side'] = (rnn_start, valid_ind, att)              # the policy hidden gets the unshifted side-band after the target pass (ref :398-403)
        # 3. target Q (no grad) ------------------------------------------------------------------------------- ref :83-103
        self.policy.eval()
        if self.discrete_env:
            self._stage_target_discrete(c, target_policy_hidden, target_hidden)
            return
        with torch.no_grad():
            pol_t = self.target_policy if (td3 and not self.use_redq) else self.policy
            # the target critic's context encoder does not depend on the action: it runs beside the policy
            tv_embedded = self._beside(lambda: self.target_values[0].embed(next_state, state, action, target_hidden, reward))
            a_mean, _, a_next, logp_next, _, _ = pol_t.forward(next_state, state, action, target_policy_hidden, reward)
            if td3:
                noise = pol_t.noise_fn(a_mean) * p.target_action_noise_std
                a_next = torch.clamp(a_mean + torch.clamp(noise, -p.target_action_noise_clip, p.target_action_noise_clip), -1, 1)
                logp_next = None
            q_next = self.target_values[0].forward(next_state, state, action, a_next, target_hidden, reward, embedded=tv_embedded())[0]
            c['target_Q'] = self._target_Q(q_next, sel, logp_next, reward, done, timeout, mask)
        self.last_target_Q = c['target_Q']

    def _stage_target_discrete(self, c, target_policy_hidden, target_hidden):
        """Discrete actions: y = r + (1 - done) gamma clamp(sum_a pi(a|s') (min_sel Q'(s', a) - alpha log pi(a|s')))
        (ref: sac_full_length_rnn_ensembleQ.py:134-151; REDQ subset + one-hot last action: sac_full_length_rnn_redq.py:52-72).
        The expectation over actions is one kernel (rorl_discrete_target_expect, which also initialises the guard); clamp /
        guard / statistics run on the same fused kernel as the continuous path."""
        batch, sel = c['batch'], c['sel']
        with torch.no_grad():
            onehot = self.policy.action2onehot(batch.action)
            lst_a = onehot if self.use_redq else batch.action                       # ref :141 (base class passes the raw index)
            # the target critic's context encoder does not depend on the action: it runs beside the policy
            tv_embedded = self._beside(lambda: self.target_values[0].embed(batch.next_state, batch.state, onehot, target_hidden,
                                                                           batch.reward))
            _, _, a_next, logp_next, _, _ = self.policy.forward(batch.next_state, batch.state, lst_a, target_policy_hidden, batch.reward)
            q_next = self.target_values[0].forward(batch.next_state, batch.state, onehot, a_next, target_hidden, batch.reward,
                                                   embedded=tv_embedded())[0]
            m = K.discrete_target_expect(q_next, sel, logp_next, self.log_sac_alpha.data, self.Q_guard.state, self._work)
            c['target_Q'] = self._target_finish(m, batch.reward, batch.done, batch.timeout, batch.mask)
        self.last_target_Q = c['target_Q']

    def _stage_critic(self, c, overlap):
        # 4. critic ------------------------------------------------------------------------------------------------ ref :105-114,261-295
        batch = c['batch']
        dev = self.device
        n_valid = self._stats[1:2]
        for v in self.values:
            v.train()
        q = self.values[0].forward(batch.state, batch.last_state, batch.last_action, batch.action, c['value_hidden'], batch.reward_input)[0]
        if self.discrete_env:                                         # Q of the action taken (ref :153-163)
            q = q.gather(-1, batch.action.long().unsqueeze(0).expand(q.shape[0], *batch.action.shape))
        E, M = q.shape[0], q[0].numel()
        dq = torch.empty((E, M), dtype=torch.float32, device=dev)
        qc, tq_c, mask_c = q.contiguous(), c['target_Q'].contiguous(), batch.mask.contiguous()
        N.call("rorl_q_loss_fwd_bwd", N.ptr(qc), N.ptr(tq_c), N.ptr(mask_c), N.ptr(n_valid),
               N.ptr(self._stats[2:3]), N.ptr(dq), N.ptr(self._work), E, M, N.stream())
        self.optimizer_value.zero_grad(detach=not overlap)
        if overlap:
            self._sync_value.begin()
        qc.backward(dq.view_as(qc))
        if overlap:
            self._sync_value.finish()
        else:
            self.value_arena.collect()
        c['mask_c'] = mask_c

    def _stage_value_step_and_actor(self, c, overlap):
        p = self.parameter
        td3 = self.base_algorithm == 'td3'
        dev = self.device
        batch, mask_c = c['batch'], c['mask_c']
        n_valid = self._stats[1:2]
        state, last_state, last_action, reward_input = batch.state, batch.last_state, batch.last_action, batch.reward_input
        self._freeze_no_grad(self.optimizer_value)
        self.optimizer_value.step(tau=p.sac_tau)   # + Polyak (ref :395)
        self._splits(refresh=('value',), invalidate=('target',))
        N.call("rorl_sumsq", N.ptr(self.value_arena.flat), self._l2_span['value'], N.ptr(self._stats[8:9]), N.ptr(self._work), N.stream())
        for v in self.values:
            v.eval()
        self.policy.train()
        rs, vi, at = c['side']
        c['policy_hidden'].set_rnn_start(rs), c['policy_hidden'].set_mask(vi), c['policy_hidden'].set_attention_concat_mask(at)
        # 5. actor + alpha ---------------------------------------------------------------------------------------- ref :116-132,405-432
        if not c['did_policy']:
            return
        if self.discrete_env:
            self._actor_discrete(c, overlap)
            return
        for w in self.value_arena.params:
            w.requires_grad_(False)
        try:
            # the critic's encoder under the actor is detached and its weights are frozen here: no graph, runs beside the policy
            v_embedded = self._beside(lambda: self.values[0].embed(state, last_state, last_action, c['value_hidden'], reward_input))
            a_mean, _, a_samp, logp, _, _ = self.policy.forward(state, last_state, last_action, c['policy_hidden'], reward_input)
            a_in = a_mean if td3 else a_samp
            qp = self.values[0].forward(state, last_state, last_action, a_in, c['value_hidden'], reward_input, detach_embedding=True,
                                        embedded=v_embedded())[0]
        finally:
            for w in self.value_arena.params:
                w.requires_grad_(True)
        E, M = qp.shape[0], qp[0].numel()
        qpc = qp.contiguous()
        dqp = torch.empty((E, M), dtype=torch.float32, device=dev)
        logp_c = None if td3 else logp.contiguous()
        dlogp = None if td3 else torch.empty(M, dtype=torch.float32, device=dev)
        N.call("rorl_actor_loss_fwd_bwd", N.ptr(qpc), N.ptr(logp_c), N.ptr(mask_c), N.ptr(n_valid),
               N.ptr(self.log_sac_alpha.data), float(self.target_entropy), 1 if self.use_redq else 0,
               N.ptr(self._stats[4:8]), N.ptr(dqp), N.ptr(dlogp), N.ptr(self._work), E, M, N.stream())
        self.optimizer_policy.zero_grad(detach=not overlap)
        if overlap:
            self._sync_policy.begin()
        if td3:
            qpc.backward(dqp.view_as(qpc))
        else:
            torch.autograd.backward([qpc, logp_c], [dqp.view_as(qpc), dlogp.view_as(logp_c)])
        if overlap:
            self._sync_policy.finish()
        else:
            self.policy_arena.collect()
        if not p.no_alpha_auto_tune:
            self.alpha_arena.grad.copy_(self._stats[7:8])
            if overlap:
                self._allreduce(self.alpha_arena.grad)

    def _actor_discrete(self, c, overlap):
        """Discrete actor: L = sum_mask sum_a pi(a|s) (alpha log pi(a|s) - agg_e Q_e(s, a)) / n_valid, agg = min (ensembleQ)
        or mean (REDQ) (ref: sac_full_length_rnn_ensembleQ.py:165-179, sac_full_length_rnn_redq.py:74-88); alpha is fixed
        for discrete action spaces (ref: sac.py:72-74).  One kernel forms the loss, stats[4:6] and d loss / d logp; the
        backward runs from logp through the categorical head (q gets no gradient: its weights are frozen and its embedding
        detached here)."""
        batch, mask_c = c['batch'], c['mask_c']
        n_valid = self._stats[1:2]
        state, last_state, last_action, reward_input = batch.state, batch.last_state, batch.last_action, batch.reward_input
        for w in self.value_arena.params:
            w.requires_grad_(False)
        try:
            # the critic's encoder under the actor is detached and its weights are frozen here: no graph, runs beside the policy
            v_embedded = self._beside(lambda: self.values[0].embed(state, last_state, last_action, c['value_hidden'], reward_input))
            _, _, a_samp, logp, _, _ = self.policy.forward(state, last_state, last_action, c['policy_hidden'], reward_input)
            qp = self.values[0].forward(state, last_state, last_action, a_samp, c['value_hidden'], reward_input,
                                        detach_embedding=True, embedded=v_embedded())[0]
        finally:
            for w in self.value_arena.params:
                w.requires_grad_(True)
        dlogp = K.discrete_actor_loss(qp, logp, mask_c, n_valid, self.log_sac_alpha.data, 1 if self.use_redq else 0,
                                      self._stats[4:6], self._work)
        self.optimizer_policy.zero_grad(detach=not overlap)
        if overlap:
            self._sync_policy.begin()
        torch.autograd.backward(logp, dlogp)
        if overlap:
            self._sync_policy.finish()
        else:
            self.policy_arena.collect()

    def _stage_policy_step(self, c):
        if not c['did_policy']:
            return
        self._freeze_no_grad(self.optimizer_policy)
        self.optimizer_policy.step()
        self._splits(invalidate=('policy',))
        N.call("rorl_sumsq", N.ptr(self.policy_arena.flat), self._l2_span['policy'], N.ptr(self._stats[9:10]), N.ptr(self._work), N.stream())
        if not self.parameter.no_alpha_auto_tune:
            self.optimizer_alpha.step()
            self.log_sac_alpha.data.clamp_(max=1.0)

    def _arm_grad_detection(self):
        """First update with weight decay on: record which parameters receive a gradient at all (hooks fire on
        accumulation), so that the fused optimizer can skip the others as torch.optim.AdamW skips `.grad is None`."""
        p = self.parameter
        if self._grad_seen is not None or not (p.policy_l2_norm > 0 or p.value_l2_norm > 0):
            return
        self._grad_seen = {}
        self._grad_hooks = [q.register_post_accumulate_grad_hook(lambda t: self._grad_seen.__setitem__(id(t), True))
                            for q in self.policy_arena.params + self.value_arena.params]

    def _freeze_no_grad(self, opt):
        if getattr(self, '_grad_hooks', None) is None:
            return
        opt.freeze_params_without_grad(self._grad_seen)
        if opt is self.optimizer_policy:                   # both models have been through their first backward
            for h in self._grad_hooks:
                h.remove()
            self._grad_hooks = None

    def _sync_guard_and_count(self):
        """Data-parallel: make n_valid and the guard state identical on every rank (SURVEY.md 8e)."""
        sync_count_and_guard(self._stats[1:2], self.Q_guard.state[0:1], self.Q_guard.state[1:2], self.dist_group)
