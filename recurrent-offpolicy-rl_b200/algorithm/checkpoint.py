"""Exact resume of a `FullLengthRNNUpdate`: the state behind `state_dict()` / `load_state_dict()` (DESIGN.md §3.14).

The update is deterministic run to run, so a run stopped after k updates and continued from its checkpoint must produce
the same bits as a run that never stopped.  That needs more than the model weights: the Adam moments and step counts, the
frozen-parameter set, log-alpha, the Q guard, the cadence counters, the cgpt dropout counters and salts, the replay buffer
and the random streams.  Everything is restored into the tensors the engine already owns (captured CUDA graphs hold
their addresses), and the graphs are kept only when nothing they bake in changed.
"""
from __future__ import annotations

from typing import Dict, List, Optional

import torch

from ..utility.rng_state import rng_state, set_rng_state

FORMAT = 1


def _named(model) -> Dict[int, str]:
    names = {}
    for n, p in model.named_parameters():
        names.setdefault(id(p), n)
    return names


def _arena_layout(arena, names: Dict[int, str]) -> List[str]:
    return [f'{names[id(p)]}:{off}:{tuple(p.shape)}' for p, off in zip(arena.params, arena.offsets)]


def _models(eng):
    return (('policy', eng.policy), ('value', eng.values[0]), ('target_value', eng.target_values[0]),
            ('target_policy', eng.target_policy))


def _attention_blocks(eng):
    """(key, module) of every attention block with a dropout counter, in a fixed order."""
    for tag, model in _models(eng):
        for mk, m in model.contextual_modules.items():
            for n, mod in m.named_modules():
                if hasattr(mod, '_drop_calls') and hasattr(mod, '_salt'):
                    yield f'{tag}.{mk}.{n}', mod


def _optimizers(eng):
    return (('policy', eng.optimizer_policy, eng.policy), ('value', eng.optimizer_value, eng.values[0]),
            ('alpha', eng.optimizer_alpha, None))


def _names_of(opt, model) -> Dict[int, str]:
    return _named(model) if model is not None else {id(opt.arena.params[0]): 'log_sac_alpha'}


def _cpu(t: torch.Tensor) -> torch.Tensor:
    return t.detach().to('cpu', copy=True)


def signature(eng) -> Dict[str, object]:
    """What a checkpoint must agree on to be loadable: anything that changes a tensor's shape or meaning."""
    def net(args, prefix):
        return {f'{prefix}.embedding_layer_type': ','.join(args['embedding_layer_type']),
                f'{prefix}.embedding_hidden': ','.join(str(w) for w in args['embedding_hidden']),
                f'{prefix}.embedding_size': int(args['embedding_size']),
                f'{prefix}.uni_model_layer_type': ','.join(args['uni_model_layer_type']),
                f'{prefix}.uni_model_hidden': ','.join(str(w) for w in args['uni_model_hidden'])}
    buf = eng.replay_buffer
    return {'algorithm': type(eng).__name__, 'discrete_env': bool(eng.discrete_env),
            'obs_dim': int(eng.policy_args['state_dim']), 'act_dim': int(eng.policy_args['action_dim']),
            'max_trajectory_len': int(eng.max_trajectory_len), 'ensemble_size': int(eng._ensemble_size),
            **net(eng.policy_args, 'policy'), **net(eng.value_args, 'value'), 'buffer_capacity': int(buf.max_transition_num),
            'buffer_row_len': int(buf.max_traj_step), 'buffer_columns': ','.join(str(w) for w in buf.column_widths())}


def _hyper_parameters(eng) -> Dict[str, object]:
    return {k: (v if isinstance(v, (bool, int, float, str)) else repr(v)) for k, v in vars(eng.parameter).items()}


def state_dict(eng) -> dict:
    torch.cuda.synchronize(eng.device)
    sd = {'format': FORMAT, 'signature': signature(eng), 'parameter': _hyper_parameters(eng)}
    for tag, model in _models(eng):
        sd[tag] = {mk: {n: _cpu(t) for n, t in msd.items()} for mk, msd in model.state_dict().items()}
    sd['layout'] = {'policy': _arena_layout(eng.policy_arena, _named(eng.policy)),
                    'value': _arena_layout(eng.value_arena, _named(eng.values[0])),
                    'target_value': _arena_layout(eng.target_arena, _named(eng.target_values[0]))}
    opts = {}
    for tag, opt, model in _optimizers(eng):
        names = _names_of(opt, model)
        opts[tag] = {'m': _cpu(opt.m), 'v': _cpu(opt.v), 'step_count': _cpu(opt.step_count),
                     'frozen': sorted(names[i] for i in opt._frozen)}
    sd['optimizers'] = opts
    pn, vn = _named(eng.policy), _named(eng.values[0])
    seen = eng._grad_seen
    sd['grad_detection'] = {'armed': seen is not None, 'hooks_live': eng._grad_hooks is not None,
                            'seen': sorted([f'policy.{pn[i]}' for i in (seen or {}) if i in pn]
                                           + [f'value.{vn[i]}' for i in (seen or {}) if i in vn])}
    sd['log_sac_alpha'] = _cpu(eng.log_sac_alpha)
    sd['q_guard'] = _cpu(eng.Q_guard.state)
    sd['stats'] = _cpu(eng._stats)
    sd['grad_num'] = int(eng.grad_num)
    sd['opt_steps'] = {k: int(v) for k, v in eng._opt_steps.items()}
    sd['guard_init_synced'] = bool(eng._guard_init_synced)
    sd['attention'] = {k: {'drop_calls': _cpu(m._drop_calls), 'salt': int(m._salt)} for k, m in _attention_blocks(eng)}
    sd['replay_buffer'] = eng.replay_buffer.state_dict()
    sd['rng'] = rng_state(eng.device)
    return sd


def _mismatch(eng, sd) -> Optional[str]:
    """First field in which the checkpoint differs structurally from the engine (None: loadable)."""
    if not isinstance(sd, dict) or sd.get('format') != FORMAT:
        got = sd.get('format') if isinstance(sd, dict) else type(sd).__name__
        return f'format (checkpoint {got!r}, this build reads {FORMAT})'
    live, saved = signature(eng), sd['signature']
    for k, v in live.items():
        if k == 'buffer_columns' and (not v or not saved.get(k)):
            continue                                 # a buffer without a trajectory yet has no column layout
        if saved.get(k) != v:
            return f'{k} (checkpoint {saved.get(k)!r}, engine {v!r})'
    bad = eng.replay_buffer.state_mismatch(sd['replay_buffer'])
    if bad is not None:
        return bad
    layouts = {'policy': _arena_layout(eng.policy_arena, _named(eng.policy)),
               'value': _arena_layout(eng.value_arena, _named(eng.values[0])),
               'target_value': _arena_layout(eng.target_arena, _named(eng.target_values[0]))}
    for tag, live_l in layouts.items():
        saved_l = list(sd['layout'][tag])
        for i in range(max(len(live_l), len(saved_l))):
            a = saved_l[i] if i < len(saved_l) else None
            b = live_l[i] if i < len(live_l) else None
            if a != b:
                return f'layout.{tag}[{i}] (checkpoint {a!r}, engine {b!r})'
    for tag, opt, _ in _optimizers(eng):
        for k in ('m', 'v'):
            if tuple(sd['optimizers'][tag][k].shape) != tuple(getattr(opt, k).shape):
                return f'optimizers.{tag}.{k}'
    for tag, model in _models(eng):
        live_sd = model.state_dict()
        if sorted(live_sd) != sorted(sd[tag]):
            return tag
        for mk, msd in live_sd.items():
            if sorted(msd) != sorted(sd[tag][mk]):
                return f'{tag}.{mk}'
            for n, t in msd.items():
                if tuple(sd[tag][mk][n].shape) != tuple(t.shape):
                    return f'{tag}.{mk}.{n}'
    live_attn = dict(_attention_blocks(eng))
    if sorted(live_attn) != sorted(sd['attention']):
        return 'attention'
    return None


def load_state_dict(eng, sd: dict) -> None:
    try:
        bad = _mismatch(eng, sd)
    except (KeyError, TypeError, AttributeError) as e:
        bad = f'missing or malformed entry {e}'
    if bad is not None:
        raise ValueError(f'checkpoint does not match this engine: {bad}')
    torch.cuda.synchronize(eng.device)
    keep_graphs = True
    with torch.no_grad():
        for tag, model in _models(eng):                 # in place: the parameters are views of the arenas
            for mk, m in model.contextual_modules.items():
                m.load_state_dict(sd[tag][mk])
        for tag, opt, model in _optimizers(eng):
            o = sd['optimizers'][tag]
            opt.m.copy_(o['m'])
            opt.v.copy_(o['v'])
            opt.step_count.copy_(o['step_count'])
            by_name = {n: i for i, n in _names_of(opt, model).items()}
            frozen = {by_name[n] for n in o['frozen']}
            if frozen != opt._frozen:                   # new lr / decay segment tables: the graphs hold the old ones
                opt._frozen = frozen
                opt._build_segments()
                keep_graphs = False
        eng.log_sac_alpha.data.copy_(sd['log_sac_alpha'])
        eng.Q_guard.state.copy_(sd['q_guard'])
        eng._stats.copy_(sd['stats'])
        for k, m in _attention_blocks(eng):
            a = sd['attention'][k]
            m._drop_calls.copy_(a['drop_calls'])
            if int(a['salt']) != m._salt:               # a Python int baked into the captured launches
                m._salt = int(a['salt'])
                keep_graphs = False
    eng.grad_num = int(sd['grad_num'])
    eng._opt_steps = {k: int(v) for k, v in sd['opt_steps'].items()}
    if bool(sd['guard_init_synced']) != eng._guard_init_synced:
        eng._guard_init_synced = bool(sd['guard_init_synced'])
        keep_graphs = False
    _restore_grad_detection(eng, sd['grad_detection'])
    eng.replay_buffer.load_state_dict(sd['replay_buffer'])
    set_rng_state(sd['rng'], eng.device)
    if not keep_graphs:
        eng.invalidate_graphs()


def _restore_grad_detection(eng, gd: dict) -> None:
    """The first-backward detection of parameters that never get a gradient (`_arm_grad_detection`): not armed, armed
    with its hooks still waiting for the policy's first backward, or finished."""
    for h in (eng._grad_hooks or []):
        h.remove()
    eng._grad_hooks = None
    if not gd['armed']:
        eng._grad_seen = None
        return
    ids = {f'policy.{n}': i for i, n in _named(eng.policy).items()}
    ids.update({f'value.{n}': i for i, n in _named(eng.values[0]).items()})
    eng._grad_seen = {ids[n]: True for n in gd['seen']}
    if gd['hooks_live']:
        eng._grad_hooks = [q.register_post_accumulate_grad_hook(lambda t: eng._grad_seen.__setitem__(id(t), True))
                           for q in eng.policy_arena.params + eng.value_arena.params]
