"""Categorical recurrent policy for discrete action spaces.

API-compatible with ContextualSACDiscretePolicy (ref: offpolicy_rnn/policy_value_models/contextual_sac_discrete_policy.py:11-141):
same constructor kwargs and registered module names; forward returns `(action_mode [..., 1], embedding,
action_sample [..., 1], log_probs [..., A], rnn_memory, full_rnn_memory)`; the probabilities are softmax(logits) mixed
with a 0.01 floor and renormalised (ref :106-111).  `sample_fn` (default: an inverse-CDF draw, see process_model_out)
is injectable; the update's losses do not depend on the sample (the discrete value ignores its action argument)."""
from typing import Optional

import torch

from .. import kernels as K
from ..models.contextual_model import ContextualModel
from ..models.RNNHidden import RNNHidden
from .contextual_sac_policy import _InputEncoders
from .utils import nearest_power_of_two, nearest_power_of_two_half


class ContextualSACDiscretePolicy(ContextualModel, _InputEncoders):
    MAX_LOG_STD = 2.0
    MIN_LOG_STD = -15.0

    def __init__(self, state_dim, action_dim, embedding_size, embedding_hidden, embedding_activations,
                 embedding_layer_type, uni_model_hidden, uni_model_activations, uni_model_layer_type, fix_rnn_length,
                 uni_model_input_mapping_dim: int = 0, reward_input=False, last_action_input=True, last_state_input=False,
                 separate_encoder=False):
        if uni_model_activations[-1] != 'linear':
            uni_model_activations = uni_model_activations[:-1] + ['linear']
        if embedding_size == 'auto':
            embedding_size = nearest_power_of_two_half(state_dim)
        if uni_model_input_mapping_dim == 'auto':
            uni_model_input_mapping_dim = nearest_power_of_two(state_dim)
        cum_dim = self._build_encoders(state_dim, action_dim, reward_input, last_action_input, last_state_input, separate_encoder)
        ContextualModel.__init__(self, embedding_input_size=cum_dim, embedding_size=embedding_size,
                                 embedding_hidden=embedding_hidden, embedding_activations=embedding_activations,
                                 embedding_layer_type=embedding_layer_type, uni_model_input_size=state_dim,
                                 uni_model_output_size=action_dim, uni_model_hidden=uni_model_hidden,
                                 uni_model_activations=uni_model_activations, uni_model_layer_type=uni_model_layer_type,
                                 fix_rnn_length=fix_rnn_length, uni_model_input_mapping_dim=uni_model_input_mapping_dim,
                                 uni_model_input_mapping_activation=embedding_activations[-1], name='ContextualSACDiscretePolicy')
        self._register_encoders()
        self.state_dim, self.action_dim = state_dim, action_dim
        self.sample_fn = None

    def forward(self, state, lst_state, lst_action, rnn_memory: Optional[RNNHidden], reward=None, detach_embedding=False):
        emb_in = self.get_embedding_input(state, lst_state, lst_action, reward)
        out, rnn_memory, emb, full = self.meta_forward(emb_in, state, rnn_memory, detach_embedding)
        action_mean, action_sample, log_probs, _ = self.process_model_out(out)
        return action_mean, emb, action_sample, log_probs, rnn_memory, full

    def process_model_out(self, model_output):
        """(mode [.., 1], sample [.., 1], log_probs [.., A], probs [.., A]) from the head output; mode and sample are int64
        action indices.  On CUDA fp32 tensors the head is one kernel forward and one backward (kernels.CategoricalHead) and
        reads nothing back to the host, so it can be graph-captured.  There, without an injected `sample_fn`, the sample is
        the kernel's inverse-CDF draw from `torch.rand` uniforms: the same distribution as torch.multinomial (what
        Categorical.sample runs on CPU tensors), but not the same sequence of samples for a given seed.  An injected
        `sample_fn(probs)` supplies the sample on every device."""
        if model_output.is_cuda and model_output.dtype == torch.float32:
            u = None if self.sample_fn is not None else torch.rand(model_output.shape[:-1], device=model_output.device)
            mode, sample, log_probs, probs = K.categorical_head(model_output, u)
            sample = self.sample_fn(probs) if self.sample_fn is not None else sample.long()
            return mode.long(), sample, log_probs, probs
        probs = (model_output - model_output.max(dim=-1, keepdim=True).values).exp()
        probs = probs / probs.sum(dim=-1, keepdim=True)
        probs = probs + 0.01                                                # exploration floor (ref :108-109)
        probs = probs / probs.sum(dim=-1, keepdim=True)
        action_mean = probs.argmax(dim=-1, keepdim=True)
        if self.sample_fn is not None:
            action_sample = self.sample_fn(probs)
        else:
            action_sample = torch.distributions.Categorical(probs=probs.detach()).sample().unsqueeze(-1)
        return action_mean, action_sample, torch.log(probs), probs

    def select_with_action(self, action: torch.Tensor, data: torch.Tensor) -> torch.Tensor:
        return data.gather(-1, action.long())

    def action2onehot(self, action: torch.Tensor):
        """F.one_hot(action.squeeze(-1).long(), num_classes=A).float(), bit for bit, built by comparison with arange(A):
        F.one_hot reads the index range back to the host, which would stall the stream and break graph capture."""
        idx = action.squeeze(-1).long().unsqueeze(-1)
        return (idx == torch.arange(self.action_dim, device=action.device)).float()

    def forward_embedding(self, state, lst_state, lst_action, rnn_memory, reward):
        return self.get_embedding(self.get_embedding_input(state, lst_state, lst_action, reward), rnn_memory)
