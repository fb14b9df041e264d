"""The process-global random streams an update draws from, as checkpoint entries that `torch.load(weights_only=True)`
accepts: numpy's global MT19937 (the replay sampler and the REDQ subset), torch's CPU generator and the CUDA generator of
one device (policy noise, TD3 target noise, categorical draws, random first hidden states)."""
import numpy as np
import torch


def numpy_state() -> dict:
    """numpy's global state without its tuple: the 624 key words as an int64 tensor plus plain ints / a float."""
    kind, keys, pos, has_gauss, cached = np.random.get_state()
    assert kind == 'MT19937', kind
    return {'keys': torch.from_numpy(np.asarray(keys, dtype=np.int64)), 'pos': int(pos), 'has_gauss': int(has_gauss),
            'cached_gaussian': float(cached)}


def set_numpy_state(sd: dict) -> None:
    np.random.set_state(('MT19937', sd['keys'].numpy().astype(np.uint32), int(sd['pos']), int(sd['has_gauss']),
                         float(sd['cached_gaussian'])))


def rng_state(device) -> dict:
    out = {'numpy': numpy_state(), 'torch_cpu': torch.get_rng_state()}
    if device is not None and torch.device(device).type == 'cuda':
        out['torch_cuda'] = torch.cuda.get_rng_state(device)
    return out


def set_rng_state(sd: dict, device) -> None:
    set_numpy_state(sd['numpy'])
    torch.set_rng_state(sd['torch_cpu'])
    if 'torch_cuda' in sd:
        torch.cuda.set_rng_state(sd['torch_cuda'], device)
