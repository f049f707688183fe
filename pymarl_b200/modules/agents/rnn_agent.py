"""RNNAgent: fc1 -> ReLU -> GRUCell -> fc2 (reference: modules/agents/rnn_agent.py:7-36).

The nn.Linear / nn.GRUCell members only hold the parameters (same names, shapes and init
as the reference, so checkpoints interchange); forward() runs the CUDA kernels
(pmb_agent_fc1_dense_fwd + pmb_agent_gru_unroll_fwd).  Inference only: the learner has its
own hand-written backward and never differentiates through this module."""
import ctypes as C
from collections import OrderedDict

import torch as th
import torch.nn as nn

from ... import _lib, flat as _flat


class RNNAgent(nn.Module):
    def __init__(self, input_shape, args):
        super().__init__()
        self.args = args
        self.input_shape = input_shape
        if isinstance(input_shape, tuple):
            assert len(input_shape) == 1, "Input shape has unsupported dimensionality: {}".format(input_shape)
            input_shape = input_shape[0]
        elif isinstance(input_shape, (dict, OrderedDict)):
            input_shape = input_shape["1d"][0]
        self.d_in = int(input_shape)
        self.fc1 = nn.Linear(self.d_in, args.rnn_hidden_dim)
        self.rnn = nn.GRUCell(args.rnn_hidden_dim, args.rnn_hidden_dim)
        self.fc2 = nn.Linear(args.rnn_hidden_dim, args.n_actions)

    def init_hidden(self):
        return self.fc1.weight.new(1, self.args.rnn_hidden_dim).zero_()

    def _dims(self, rows):
        a = self.args
        # dense input: the kernel only needs H, A and D_in = O + A*last_action + N*agent_id
        return _lib.make_dims(B=rows, T=1, N=1, O=self.d_in, S=1, A=a.n_actions, H=a.rnn_hidden_dim, E=1,
                              obs_last_action=False, obs_agent_id=False, mixer=None)

    @th.no_grad()
    def forward(self, inputs, hidden_state):
        if isinstance(inputs, (dict, OrderedDict)):
            inputs = inputs["1d"]
        _lib.require_cuda(inputs, "inputs")
        H, A = self.args.rnn_hidden_dim, self.args.n_actions
        x_in = inputs.reshape(-1, self.d_in).to(th.float32).contiguous()
        rows = x_in.shape[0]
        h_in = hidden_state.reshape(-1, H)
        if h_in.shape[0] != rows:
            h_in = h_in.expand(rows, H)
        h_in = h_in.to(th.float32).contiguous()
        dims = self._dims(rows)
        flat = C.c_void_p(_flat.ensure_block(self, "agent", dims))
        x = th.empty(rows, H, dtype=th.float32, device=x_in.device)
        q = th.empty(rows, A, dtype=th.float32, device=x_in.device)
        h = th.empty(rows, H, dtype=th.float32, device=x_in.device)
        # H = 128 computes the input gates of all rows as one GEMM before the recurrence: they need a buffer
        gates = th.empty(rows, 4 * H, dtype=th.float32, device=x_in.device) if H == 128 else None
        s = _lib.stream_ptr(x_in.device)
        L = _lib.lib()
        _lib.check(L.pmb_agent_fc1_dense_fwd(C.byref(dims), rows, self.d_in, _lib.ptr(x_in), flat,
                                             _lib.ptr(x), s), "pmb_agent_fc1_dense_fwd")
        _lib.check(L.pmb_agent_gru_unroll_fwd(C.byref(dims), rows, 1, flat, _lib.ptr(x), _lib.ptr(h_in),
                                              None, _lib.ptr(gates), _lib.ptr(q), _lib.ptr(h), s), "pmb_agent_gru_unroll_fwd")
        return q, h
