"""RNNAgent: fc1 -> ReLU -> GRUCell -> fc2 (reference: modules/agents/rnn_agent.py:7-36).

The nn.Linear / nn.GRUCell members only hold the parameters (same names, shapes and init
as the reference, so checkpoints interchange); forward() runs the CUDA kernels
(pmb_agent_fc1_dense_fwd + pmb_agent_gru_unroll_fwd).

By default the module is inference only (its outputs carry no graph): the built-in learners own hand-written backward
passes.  With ``args.autograd_modules = True`` and grad mode on, forward() is one autograd node (AgentStep): gradients
reach the eight parameters and the hidden state through pmb_agent_step_bwd, for learners that call loss.backward().
That mode runs the fp32 kernels whatever ``args.precision`` says."""
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

    def forward(self, inputs, hidden_state):
        if isinstance(inputs, (dict, OrderedDict)):
            inputs = inputs["1d"]
        _lib.require_cuda(inputs, "inputs")
        if _lib.autograd_mode(self.args):
            if inputs.requires_grad:
                raise _lib.PmbError("RNNAgent: no gradient flows into the agent inputs (batch data); pass inputs.detach()")
            H = self.args.rnn_hidden_dim
            x_in = inputs.detach().reshape(-1, self.d_in).to(th.float32).contiguous()
            rows = x_in.shape[0]
            h_in = hidden_state.reshape(-1, H)
            if h_in.shape[0] != rows:
                h_in = h_in.expand(rows, H)
            h_in = h_in.to(th.float32).contiguous()
            return AgentStep.apply(self, self._dims(rows), (None, 0, [x_in]), h_in, *self.parameters())
        with th.no_grad():
            return self._forward_inference(inputs, hidden_state)

    def _forward_inference(self, inputs, hidden_state):
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


class AgentStep(th.autograd.Function):
    """One agent step as one autograd node: fc1 (pmb_agent_fc1_fwd on the batch at time t, or pmb_agent_fc1_dense_fwd on
    a dense input matrix) and pmb_agent_gru_unroll_fwd with nt = 1, saving x, (h_prev | h) and the gates; the backward is
    pmb_agent_step_bwd.  src = (pmb_batch, t, [tensors the batch points into]) or (None, 0, [dense inputs [rows][D_in]]).
    Returns q [rows][A] and h [rows][H]; gradients flow to h_in and to the parameters (named_parameters() order).
    Everything the backward reads is a saved tensor, so it is freed with the graph's buffers after the backward."""

    @staticmethod
    def forward(ctx, agent, dims, src, h_in, *params):
        batch, t, tensors = src
        rows, H, A = h_in.shape[0], dims.H, dims.A
        flat = C.c_void_p(_flat.ensure_block(agent, "agent", dims))
        dev = h_in.device
        x = th.empty(rows, H, dtype=th.float32, device=dev)
        h_stash = th.empty(2, rows, H, dtype=th.float32, device=dev)
        gates = th.empty(rows, 4 * H, dtype=th.float32, device=dev)
        q = th.empty(rows, A, dtype=th.float32, device=dev)
        h = th.empty(rows, H, dtype=th.float32, device=dev)
        s = _lib.stream_ptr(dev)
        L = _lib.lib()
        if batch is not None:
            _lib.check(L.pmb_agent_fc1_fwd(C.byref(dims), C.byref(batch), t, 1, flat, _lib.ptr(x), s), "pmb_agent_fc1_fwd")
        else:
            _lib.check(L.pmb_agent_fc1_dense_fwd(C.byref(dims), rows, dims.O, _lib.ptr(tensors[0]), flat, _lib.ptr(x), s),
                       "pmb_agent_fc1_dense_fwd")
        _lib.check(L.pmb_agent_gru_unroll_fwd(C.byref(dims), rows, 1, flat, _lib.ptr(x), _lib.ptr(h_in), _lib.ptr(h_stash),
                                              _lib.ptr(gates), _lib.ptr(q), _lib.ptr(h), s), "pmb_agent_gru_unroll_fwd")
        # the parameters too: an in-place update before the backward raises
        ctx.save_for_backward(x, h_stash, gates, *tensors, *params)
        ctx.set_materialize_grads(False)
        ctx.step = (agent, dims, batch, t, flat)
        return q, h

    @staticmethod
    def backward(ctx, dq, dh):
        _lib.no_double_backward("RNNAgent")
        agent, dims, batch, t, flat = ctx.step
        saved = ctx.saved_tensors                             # also keeps alive (and version-checks) what `batch` points into
        x, h_stash, gates = saved[:3]
        inputs = saved[3] if batch is None else None
        rows, dev = x.shape[0], x.device
        dq = None if dq is None else dq.to(th.float32).contiguous()
        dh = None if dh is None else dh.to(th.float32).contiguous()
        dh_prev = th.empty(rows, dims.H, dtype=th.float32, device=dev) if ctx.needs_input_grad[3] else None
        layout = _lib.flat_layout(dims)
        g = th.empty(_flat.block_numel(layout, "agent"), dtype=th.float32, device=dev)
        L = _lib.lib()
        nbytes = L.pmb_agent_step_bwd_workspace_bytes(C.byref(dims), rows)
        scratch = th.empty(max(nbytes, 1), dtype=th.uint8, device=dev)
        _lib.check(L.pmb_agent_step_bwd(C.byref(dims), None if batch is None else C.byref(batch), t, _lib.ptr(inputs), rows,
                                        flat, _lib.ptr(x), _lib.ptr(h_stash), _lib.ptr(gates), _lib.ptr(dq), _lib.ptr(dh),
                                        _lib.ptr(dh_prev), _lib.ptr(g), _lib.ptr(scratch), nbytes, _lib.stream_ptr(dev)),
                   "pmb_agent_step_bwd")
        grads = [gv if need else None for gv, need in zip(_flat.grad_views(g, layout, agent, "agent"), ctx.needs_input_grad[4:])]
        return (None, None, None, dh_prev) + tuple(grads)
