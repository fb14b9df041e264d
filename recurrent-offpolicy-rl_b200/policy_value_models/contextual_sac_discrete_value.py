"""Recurrent ensemble-Q value model for discrete action spaces: one Q per action from (state, context embedding).

API-compatible with ContextualSACDiscreteValue (ref: offpolicy_rnn/policy_value_models/contextual_sac_discrete_value.py:9-135):
with `separate_encoder` the universal network sees act(Linear(state)) registered as `state_input_encoder_q` (ref :50-56,
:98-102); the `action` argument of forward is accepted and ignored, as in the reference (ref :119-126).
forward returns `(Q [E, B, L, A], embedding, rnn_memory, full_rnn_memory)`."""
from typing import Optional

import torch

from ..models.contextual_model import ContextualModel
from ..models.linear import Linear
from ..models.RNNHidden import RNNHidden
from ..models.rnn_base import ACTIVATIONS
from .contextual_sac_policy import _InputEncoders
from .utils import nearest_power_of_two, nearest_power_of_two_half


class ContextualSACDiscreteValue(ContextualModel, _InputEncoders):
    def __init__(self, state_dim, action_dim, embedding_size, embedding_hidden, embedding_activations,
                 embedding_layer_type, uni_model_hidden, uni_model_activations, uni_model_layer_type, fix_rnn_length,
                 uni_model_input_mapping_dim: int = 0, reward_input=False, last_action_input=True, last_state_input=False,
                 separate_encoder=False):
        self.embedding_state_dim = state_dim
        if embedding_size == 'auto':
            embedding_size = nearest_power_of_two_half(state_dim)
        if uni_model_input_mapping_dim == 'auto':
            uni_model_input_mapping_dim = nearest_power_of_two(state_dim + action_dim)
        cum_dim = self._build_encoders(state_dim, action_dim, reward_input, last_action_input, last_state_input, separate_encoder)
        uni_in = state_dim
        self.state_input_encoder = torch.nn.Identity()
        if uni_model_input_mapping_dim > 0 and separate_encoder:
            self.state_input_encoder = Linear(state_dim, uni_model_input_mapping_dim)
            uni_in = uni_model_input_mapping_dim
            uni_model_input_mapping_dim = 0
        ContextualModel.__init__(self, embedding_input_size=cum_dim, embedding_size=embedding_size,
                                 embedding_hidden=embedding_hidden, embedding_activations=embedding_activations,
                                 embedding_layer_type=embedding_layer_type, uni_model_input_size=uni_in,
                                 uni_model_output_size=action_dim, uni_model_hidden=uni_model_hidden,
                                 uni_model_activations=uni_model_activations, uni_model_layer_type=uni_model_layer_type,
                                 fix_rnn_length=fix_rnn_length, uni_model_input_mapping_dim=uni_model_input_mapping_dim,
                                 uni_model_input_mapping_activation=embedding_activations[-1], name='ContextualSACValue')
        self.uni_model_input_mapping_activation_func = ACTIVATIONS[embedding_activations[-1]]()
        self._register_encoders()
        if separate_encoder:
            self.contextual_register_rnn_base_module(self.state_input_encoder, 'state_input_encoder_q')
        self.state_dim, self.action_dim = state_dim, action_dim

    def state_encoding(self, state):
        if self.separate_encoder:
            return self.uni_model_input_mapping_activation_func(self.state_input_encoder(state))
        return self.state_input_encoder(state)

    def forward(self, state, lst_state, lst_action, action, rnn_memory: Optional[RNNHidden], reward, detach_embedding=False,
                embedded=None):
        """embedded: what `embed(...)` returned for the same (state, lst_state, lst_action, rnn_memory, reward), so that a
        caller may run the context encoder ahead of (or beside) the policy, as for the continuous value."""
        emb_in = None if embedded is not None else self.get_embedding_input(state, lst_state, lst_action, reward)
        value, rnn_memory, emb, full = self.meta_forward(emb_in, self.state_encoding(state), rnn_memory, detach_embedding,
                                                         embedded=embedded)
        return value, emb, rnn_memory, full

    def embed(self, state, lst_state, lst_action, rnn_memory: Optional[RNNHidden], reward):
        """The context-encoder half of forward(): (embedding, its hidden, its per-layer record)."""
        return self._meta_forward_embedding(self.get_embedding_input(state, lst_state, lst_action, reward), rnn_memory)

    def forward_embedding(self, state, lst_state, lst_action, rnn_memory, reward):
        return self.get_embedding(self.get_embedding_input(state, lst_state, lst_action, reward), rnn_memory)
