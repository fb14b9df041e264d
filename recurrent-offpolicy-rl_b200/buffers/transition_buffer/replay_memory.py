"""Flat transition ring buffer (host float64 master copy + device fp32 mirror).

Keeps the reference's storage contract (ref: offpolicy_rnn/buffers/transition_buffer/replay_memory.py):
`Transition` field order (:11), one row per transition with `None` fields taking no columns (:154-177),
whole trajectories appended when `done` arrives (:213-234), oldest trajectories evicted when over
capacity (:189-199), the write pointer wrapping only between trajectories (:209-210), and
`_traj_ind_sample`'s use of the numpy GLOBAL RNG (:56-90), which parity depends on.

B200-native part: every completed trajectory is also written (as fp32, the dtype `n2t` casts to,
ref: offpolicy_rnn/utility/sample_utility.py:30-31) into a device-resident ring, so that sampling is a
device gather and no per-update host->device copy of the batch exists.
"""
from __future__ import annotations

from collections import namedtuple
from typing import Dict, List, Optional

import numpy as np
import torch

tuplenames = ('state', 'last_state', 'last_action', 'action', 'next_state', 'reward', 'logp', 'mask', 'start', 'done',
              'reward_input', 'timeout')
Transition = namedtuple('Transition', tuplenames)


def _width(item) -> int:
    if isinstance(item, np.ndarray):
        return item.shape[-1]
    if isinstance(item, list):
        return len(item)
    if item is None:
        return 0
    if np.isscalar(item):
        return 1
    raise NotImplementedError(f'not implement for type of {type(item)}')


def _encode_pending(memory: List[Transition]) -> dict:
    """The partial trajectory `mem_push` collects until `done`, one float64 tensor per field stacked over the steps.
    Fields given as Python / numpy scalars come back as Python floats, arrays and lists as float64 arrays: either way
    they land in the buffer as the same float64 row."""
    out = {'steps': len(memory)}
    for i, name in enumerate(tuplenames):
        vals = [t[i] for t in memory]
        if all(v is None for v in vals):
            continue
        if any(v is None for v in vals):
            raise ValueError(f'pending trajectory: field {name} is None in some steps only')
        out[name] = torch.from_numpy(np.stack([np.asarray(v, dtype=np.float64) for v in vals]))
        out[name + '.scalar'] = all(np.isscalar(v) for v in vals)
    return out


def _decode_pending(sd: dict) -> List[Transition]:
    fields = []
    for name in tuplenames:
        if name not in sd:
            fields.append([None] * sd['steps'])
        elif sd[name + '.scalar']:
            fields.append([float(x) for x in sd[name].tolist()])
        else:
            fields.append(list(sd[name].numpy()))
    return [Transition(*[f[t] for f in fields]) for t in range(sd['steps'])]


class MemoryArray(object):
    def __init__(self, max_transition_num: int = 1000000, max_traj_step: Optional[int] = 1000, rnn_slice_length=1,
                 device: Optional[torch.device] = None):
        self.max_transition_num = int(max_transition_num)
        self.max_traj_step = max_traj_step
        self.rnn_slice_length = rnn_slice_length
        self.device = device
        self.memory: List[Transition] = []
        self.trajectory_length: List[int] = []
        self.trajectory_start: List[int] = []
        self.memory_buffer: Optional[np.ndarray] = None      # host float64, reference layout
        self.device_buffer: Optional[torch.Tensor] = None    # device fp32 mirror
        self.ind_range: Optional[List[List[int]]] = None
        self.name2range: Dict[str, List[int]] = {}
        self.ptr = 0
        self.transition_count = 0

    # ---- bookkeeping ----------------------------------------------------------------------------------
    @property
    def available_traj_num(self):
        return len(self.trajectory_length)

    def __len__(self):
        return len(self.trajectory_length)

    @property
    def size(self):
        return self.transition_count

    def reset(self):
        self.memory, self.trajectory_length, self.trajectory_start = [], [], []
        self.ptr = self.transition_count = 0

    def _init_memory_buffer(self, transition: Transition):
        col = 0
        self.ind_range = []
        for name, item in zip(tuplenames, transition):
            w = _width(item)
            self.ind_range.append(list(range(col, col + w)))
            self.name2range[name] = self.ind_range[-1]
            col += w
        rows = int(self.max_transition_num + self.max_traj_step)
        self.memory_buffer = np.zeros((rows, col))
        if self.device is not None and torch.device(self.device).type == 'cuda':
            self.device_buffer = torch.zeros((rows, col), dtype=torch.float32, device=self.device)

    def transition_to_array(self, transition: Transition) -> np.ndarray:
        parts = []
        for item in transition:
            if isinstance(item, np.ndarray):
                parts.append(item.reshape((1, -1)))
            elif isinstance(item, list):
                parts.append(np.array(item).reshape((1, -1)))
            elif item is None:
                continue
            elif np.isscalar(item):
                parts.append(np.array([[item]]))
            else:
                raise NotImplementedError(f'not implement for type of {type(item)}')
        row = np.hstack(parts)
        assert row.shape[-1] == self.memory_buffer.shape[-1], f'data_size: {row.shape}, buffer_size: {self.memory_buffer.shape}'
        return row

    def array_to_transition(self, data) -> Transition:
        return Transition(*[data[..., r[0]:r[-1] + 1] if len(r) else None for r in self.ind_range])

    # ---- insertion ---------------------------------------------------------------------------------------
    def _evict_for(self, traj_len: int):
        drop = 0
        if self.transition_count + traj_len > self.max_transition_num:
            c = self.transition_count
            while c + traj_len > self.max_transition_num:
                c -= self.trajectory_length[drop]
                drop += 1
        if drop:
            self.transition_count -= sum(self.trajectory_length[:drop])
            del self.trajectory_start[:drop]
            del self.trajectory_length[:drop]

    def complete_traj(self, memory: List[Transition]):
        if self.memory_buffer is None:
            self._init_memory_buffer(memory[0])
        self.push_trajectory_array(np.vstack([self.transition_to_array(t) for t in memory]))

    def push_trajectory_array(self, rows: np.ndarray):
        """Append one whole trajectory given as a [T, F] float64 array in buffer column order (bulk form of
        the per-transition loop at ref :201-208)."""
        n = rows.shape[0]
        self._evict_for(n)
        self.trajectory_start.append(self.ptr)
        self.memory_buffer[self.ptr:self.ptr + n] = rows
        if self.device_buffer is not None:
            self.device_buffer[self.ptr:self.ptr + n].copy_(torch.from_numpy(rows).to(torch.float32), non_blocking=True)
        self.ptr += n
        self.trajectory_length.append(n)
        self.transition_count += n
        if self.ptr >= self.max_transition_num:
            self.ptr = 0

    def mem_push(self, transition: Transition, parallel_num=1, valid_data=True):
        if not valid_data:
            self.memory = []
            return
        self.memory.append(transition)
        done = transition.done if np.isscalar(transition.done) else np.array(transition.done)
        mask = transition.mask if np.isscalar(transition.mask) else np.array(transition.mask)
        if np.all(done):
            if np.all(mask):
                if parallel_num == 1:
                    self.complete_traj(self.memory)
                else:
                    for i in range(parallel_num):
                        self.complete_traj([Transition(*[f[i] if (f is not None and not np.isscalar(f)) else f for f in t])
                                            for t in self.memory])
            self.memory = []

    # ---- checkpoint state ---------------------------------------------------------------------------------------
    def column_widths(self) -> List[int]:
        """Columns per `Transition` field, in field order ([] before the first trajectory fixes the layout)."""
        return [len(r) for r in self.ind_range] if self.ind_range is not None else []

    def state_dict(self) -> dict:
        """Everything that decides what the buffer holds and what the sampler draws from it, as tensors / ints / strings
        (`torch.load(weights_only=True)` reads it back): the host rows up to the end of the highest live trajectory (rows
        above it are never read), the trajectory start / length lists, the write pointer, the transition count and the
        pending partial trajectory.  The device mirror is not stored: it is the fp32 cast of the host rows."""
        end = max((s + n for s, n in zip(self.trajectory_start, self.trajectory_length)), default=0)
        rows = self.memory_buffer[:end] if self.memory_buffer is not None else np.zeros((0, 0))
        return {'max_transition_num': self.max_transition_num, 'max_traj_step': int(self.max_traj_step),
                'columns': self.column_widths(), 'rows': torch.from_numpy(np.array(rows, dtype=np.float64)),
                'trajectory_start': torch.tensor(self.trajectory_start, dtype=torch.int64),
                'trajectory_length': torch.tensor(self.trajectory_length, dtype=torch.int64),
                'ptr': int(self.ptr), 'transition_count': int(self.transition_count), 'pending': _encode_pending(self.memory)}

    def state_mismatch(self, sd: dict) -> Optional[str]:
        """Name of the first structural field in which `sd` differs from this buffer, or None.  A buffer that has not seen
        a trajectory yet takes any column layout."""
        for k in ('max_transition_num', 'max_traj_step'):
            if int(sd[k]) != int(getattr(self, k)):
                return f'replay_buffer.{k}'
        if sd['columns'] and self.ind_range is not None and list(sd['columns']) != self.column_widths():
            return 'replay_buffer.columns'
        return None

    def load_state_dict(self, sd: dict) -> None:
        """Restore what `state_dict()` saved.  The host and device buffers are kept (allocated from the saved column
        layout if this buffer has none yet); the device rows are rewritten from the host rows with one copy."""
        bad = self.state_mismatch(sd)
        if bad is not None:
            raise ValueError(f'replay-buffer state does not match this buffer: {bad}')
        if sd['columns'] and self.memory_buffer is None:
            self._init_memory_buffer(Transition(*[np.zeros(w) if w else None for w in sd['columns']]))
        rows = sd['rows'].numpy()
        end = rows.shape[0]
        if end:
            self.memory_buffer[:end] = rows
            if self.device_buffer is not None:
                self.device_buffer[:end].copy_(torch.from_numpy(rows.astype(np.float32)))
        self.trajectory_start = [int(x) for x in sd['trajectory_start'].tolist()]
        self.trajectory_length = [int(x) for x in sd['trajectory_length'].tolist()]
        self.ptr, self.transition_count = int(sd['ptr']), int(sd['transition_count'])
        self.memory = _decode_pending(sd['pending'])

    # ---- trajectory index draw (numpy global RNG; call order is part of the parity contract) ----------------
    def _traj_ind_sample(self, batch_size, max_sample_size) -> np.ndarray:
        n_traj = self.available_traj_num
        mean_len = self.transition_count / n_traj
        want = int(np.ceil(batch_size / mean_len)) if batch_size is not None else n_traj
        max_traj_num = None
        if max_sample_size is not None:
            max_traj_num = int(np.ceil(max_sample_size / self.max_traj_step))
            want = min(want, max_traj_num)
        perm = np.random.permutation(n_traj)
        if batch_size is None:
            inds = np.arange(n_traj)
        elif want <= n_traj:
            inds = perm[:int(want)]
        else:
            inds = np.random.randint(0, n_traj, (int(want),))
        total = sum(self.trajectory_length[i] for i in inds)
        count = len(inds)
        extra = []
        while total < batch_size and (max_sample_size is None or count < max_traj_num):
            count += 1
            pos = want + len(extra)
            idx = perm[pos] if n_traj > pos else np.random.randint(low=0, high=n_traj)
            total += self.trajectory_length[idx]
            extra.append(idx)
        if extra:
            inds = np.concatenate((inds, np.array(extra)), axis=0)
        return inds
