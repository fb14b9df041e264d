"""The policy acting for a batch of environments: one CUDA-graph replay per environment step.

In the reference's `train()` loop every environment step runs `policy.forward` at L = 1 with the hidden state carried
over (ref: algorithm/sac.py rollout).  Eagerly that is several dozen launches plus Python per step.  `PolicyActor` owns
static device buffers (packed inputs, every layer's carried hidden state, packed outputs) and replays one captured
graph of that forward per step:

    pinned H2D copy of the inputs -> graph replay (reset rows zeroed, policy.forward at L = 1 under no_grad with its
    head and in-graph noise / uniforms, new hidden state copied back) -> D2H copy into pinned memory -> one event wait

The first call runs eagerly (warm-up: cluster occupancy queries, library heuristics); the second captures.  The graph
reads the policy's parameters in place, so it stays valid across `train_one_batch()` and `load_state_dict()`; when the
engine rebuilds its arenas (`load_models()`, `_finalize_models()`) its `model_generation` changes and the actor
recaptures.  Everything runs on the current stream, ordered with the update.
"""
from __future__ import annotations

import numpy as np
import torch

from .. import _native as N
from ..models.RNNHidden import RNNHidden
from ..policy_value_models.contextual_td3_policy import ContextualTD3Policy


def _graph_safe(fn, default) -> bool:
    return fn is None or fn is default or getattr(fn, 'graph_safe', False)


class PolicyActor:
    """`step(state, last_state, last_action, reward, start)` for `n_envs` environments stepped in lockstep.

    Inputs are host arrays with `n_envs` rows: state [S], last_state [S] (if the policy takes it), last_action [the
    policy's last-action width: the action for continuous policies, the one-hot row for discrete ones] (if it takes it),
    reward [1] (if it takes it), start [1] (1 = the environment begins an episode: its hidden rows are zeroed before the
    step, the same as starting from `make_init_state`).  Inputs the policy does not take may be None.

    Returns numpy arrays of what `policy.forward` returns for acting at L = 1, one row per environment:
      continuous (SAC / TD3): (action_mean [n, A], action_sample [n, A], log_prob [n, 1]; TD3: zeros [n, A])
      discrete:               (action_mode [n, 1] int64, action_sample [n, 1] int64, log_probs [n, A])
    """

    def __init__(self, policy, n_envs: int, generation=None, use_cuda_graph: bool = True):
        layer_types = list(policy.embedding_network.layer_type) + list(policy.uni_network.layer_type)
        if any(str(t).startswith(('cgpt', 'gpt', 'transformer')) for t in layer_types):
            raise NotImplementedError(
                'make_actor: the cgpt encoder keeps its kv-cache position (seqlen_offset) on the host, one position for the '
                'whole batch, so environments that reset independently cannot share one captured step')
        dev = torch.device(policy.device)
        if dev.type != 'cuda':
            raise RuntimeError('the actor runs on sm_100a kernels only; no CPU path exists')
        if int(n_envs) < 1:
            raise ValueError(f'n_envs must be >= 1, got {n_envs}')
        self.policy, self.n_envs, self.device = policy, int(n_envs), dev
        self._generation = generation if generation is not None else (lambda: 0)
        self.use_cuda_graph = bool(use_cuda_graph)
        self.discrete = not hasattr(policy, 'noise_fn')
        S = policy.state_dim
        self._widths = [('state', S), ('last_state', policy.last_obs_dim), ('last_action', policy.last_act_dim),
                        ('reward', policy.reward_dim), ('start', 1)]
        n, W = self.n_envs, sum(w for _, w in self._widths)
        self._in_host = torch.zeros((n, W), dtype=torch.float32).pin_memory()
        self._in_dev = torch.zeros((n, W), dtype=torch.float32, device=dev)
        self._views, off = {}, 0
        for name, w in self._widths:
            self._views[name] = (off, w)
            off += w
        A = policy.action_dim
        # TD3's log-prob placeholder is zeros shaped like the action
        self._out_cols = [1, 1, A] if self.discrete else [A, A, A if isinstance(policy, ContextualTD3Policy) else 1]
        self._out_dev = torch.zeros((n, sum(self._out_cols)), dtype=torch.float32, device=dev)
        self._out_host = torch.zeros_like(self._out_dev, device='cpu').pin_memory()
        init = policy.make_init_state(n, dev)
        self.hidden = RNNHidden(len(init), init._rnn_types, dev)       # static carried state (no zero-state marks)
        for s in init._data:
            self.hidden.append(tuple(t.clone() for t in s) if isinstance(s, tuple) else s.clone())
        self._event = torch.cuda.Event()
        self._graph = None
        self._graph_gen = None
        self._launches = 0
        self._eager_calls = 0

    # ---- the captured body -----------------------------------------------------------------------------------
    def _col(self, name):
        off, w = self._views[name]
        return None if w == 0 else self._in_dev[:, off:off + w].unsqueeze(1)         # [n, 1, w]

    def _body(self):
        starting = (self._in_dev[:, -1] > 0.5).view(1, -1, 1)                          # environments beginning an episode
        for s in self.hidden._data:
            for t in (s if isinstance(s, tuple) else (s,)):
                t.masked_fill_(starting, 0.0)
        with torch.no_grad():
            out = self.policy.forward(self._col('state'), self._col('last_state'), self._col('last_action'), self.hidden,
                                      reward=self._col('reward'))
            new = out[4]
            for dst, src in zip(self.hidden._data, new._data):
                if isinstance(dst, tuple):
                    for d, s in zip(dst, src):
                        if d is not s:
                            d.copy_(s.reshape(d.shape))
                elif dst is not src:
                    dst.copy_(src.reshape(dst.shape))
            off = 0
            for t, w in zip((out[0], out[2], out[3]), self._out_cols):
                self._out_dev[:, off:off + w].copy_(t.reshape(self.n_envs, w))
                off += w

    def _capturable(self) -> bool:
        if not self.use_cuda_graph:
            return False
        if self.discrete:
            return _graph_safe(self.policy.sample_fn, None)
        return _graph_safe(self.policy.noise_fn, torch.randn_like)

    # ---- public API ----------------------------------------------------------------------------------------------
    def reset(self) -> None:
        """Zero every environment's hidden state."""
        for s in self.hidden._data:
            for t in (s if isinstance(s, tuple) else (s,)):
                t.zero_()

    def _pack(self, state, last_state, last_action, reward, start):
        host = self._in_host.numpy()
        given = dict(state=state, last_state=last_state, last_action=last_action, reward=reward, start=start)
        for name, (off, w) in self._views.items():
            if w == 0:
                continue
            v = given[name]
            if v is None:
                if name != 'start':
                    raise ValueError(f'PolicyActor.step: the policy takes `{name}` ({w} columns per environment)')
                host[:, off:off + w] = 0.0
                continue
            host[:, off:off + w] = np.asarray(v, dtype=np.float32).reshape(self.n_envs, w)

    def step(self, state, last_state=None, last_action=None, reward=None, start=None):
        self._pack(state, last_state, last_action, reward, start)
        self._in_dev.copy_(self._in_host, non_blocking=True)
        gen = self._generation()
        if self._graph is not None and self._graph_gen != gen:
            self._graph, self._eager_calls = None, 0                  # the arenas moved: the graph reads stale addresses
        if self._graph is not None:
            self._graph.replay()
            N.add_launches(self._launches)
        elif self._capturable() and self._eager_calls >= 1:
            # capture records the launches without running them: replay once for this step
            graph = torch.cuda.CUDAGraph()
            l0 = N.launch_count()
            with torch.cuda.graph(graph, capture_error_mode="thread_local"):
                self._body()
            self._launches = N.launch_count() - l0
            self._graph, self._graph_gen = graph, gen
            graph.replay()
            N.add_launches(self._launches)
        else:
            self._body()
            self._eager_calls += 1
        self._out_host.copy_(self._out_dev, non_blocking=True)
        self._event.record()
        self._event.synchronize()
        out = self._out_host.numpy()
        a, b, c = self._out_cols
        r0, r1, r2 = out[:, :a].copy(), out[:, a:a + b].copy(), out[:, a + b:a + b + c].copy()
        if self.discrete:
            return r0.astype(np.int64), r1.astype(np.int64), r2
        return r0, r1, r2

    @property
    def captured(self) -> bool:
        return self._graph is not None
