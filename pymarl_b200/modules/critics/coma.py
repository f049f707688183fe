"""COMACritic: the centralised counterfactual critic (reference: modules/critics/coma.py:6-59).

Parameters keep the reference names (fc1, fc2, fc3).  forward(batch, t) runs pmb_coma_critic_fwd: the input
[state | obs | other agents' actions | everyone's last actions | agent id] (coma.py:29-50) is generated on the device from
`actions` / `filled` - `actions_onehot` is never read - followed by the three dense layers.

By default the output carries no graph: the built-in COMALearner owns the training step (pmb_coma_train_step).  With
``args.autograd_modules = True`` and grad mode on, each forward call is one autograd node (CriticStep) whose backward
reaches the six parameters through pmb_coma_critic_step_bwd, for actor-critic learners of the user's own that call
loss.backward() on a loss of q.  No gradient flows into the batch.  fp32 kernels whatever ``args.precision`` says."""
import ctypes as C

import numpy as np
import torch as th
import torch.nn as nn

from ... import _lib, flat as _flat

CRITIC_KEYS = ["fc1.weight", "fc1.bias", "fc2.weight", "fc2.bias", "fc3.weight", "fc3.bias"]


def _as_int(v):
    return int(np.prod(v)) if not isinstance(v, int) else v


class COMACritic(nn.Module):
    HIDDEN = 128

    def __init__(self, scheme, args):
        super().__init__()
        self.args = args
        self.n_actions = args.n_actions
        self.n_agents = args.n_agents
        self.state_dim = _as_int(scheme["state"]["vshape"])
        self.obs_dim = _as_int(scheme["obs"]["vshape"])
        input_shape = self._get_input_shape(scheme)
        self.output_type = "q"
        self.fc1 = nn.Linear(input_shape, self.HIDDEN)
        self.fc2 = nn.Linear(self.HIDDEN, self.HIDDEN)
        self.fc3 = nn.Linear(self.HIDDEN, self.n_actions)
        self._ws = None

    def _get_input_shape(self, scheme):
        # state + observation + actions and last actions of every agent + agent id (coma.py:52-59); unlike the reference this
        # also accepts the tuple the fork's BasicMAC turns scheme["obs"]["vshape"] into (basic_controller.py:139-144)
        return self.state_dim + self.obs_dim + self.n_actions * self.n_agents * 2 + self.n_agents

    def dims(self, B, T):
        a = self.args
        return _lib.make_dims(B=B, T=max(T, 2), N=self.n_agents, O=self.obs_dim, S=self.state_dim, A=self.n_actions,
                              H=a.rnn_hidden_dim, E=self.HIDDEN, mixer=None)

    def flat_params(self):
        f = getattr(self, "_pmb_flat", None)
        if f is None or not _flat.is_bound_in_order(self, CRITIC_KEYS, f):
            _lib.require_cuda(self.fc1.weight, "critic parameters (call .cuda())")
            f = _flat.bind_in_order(self, CRITIC_KEYS)
        return f

    def _workspace(self, d, dev):
        need = _lib.lib().pmb_coma_workspace_bytes(C.byref(d))
        if self._ws is None or self._ws.numel() < need or self._ws.device != dev:
            self._ws = th.empty(need, dtype=th.uint8, device=dev)
        return self._ws, need

    def forward(self, batch, t=None):
        """-> q [B, T, N, A] (t None) or [B, 1, N, A]."""
        B, T = batch.batch_size, batch.max_seq_length
        flat = self.flat_params()
        dev = flat.device
        keep = []
        zero = th.zeros(1, device=dev)
        fields = {k: batch[k] if batch[k].is_cuda else batch[k].to(dev) for k in ("obs", "state", "actions", "filled")}
        avail = batch["avail_actions"]
        fields.update(avail_actions=avail if avail.is_cuda else avail.to(dev), reward=zero, terminated=zero.to(th.uint8))
        pb = _lib.make_batch(fields, need_state=True, keep=keep)
        if T < 2:
            raise _lib.PmbError("COMACritic needs an episode batch with at least 2 timesteps")
        d = self.dims(B, T)
        t0, nt = (0, T) if t is None else (int(t), 1)
        if _lib.autograd_mode(self.args):
            return CriticStep.apply(self, d, (pb, keep, flat), t0, nt, *self.parameters())
        with th.no_grad():
            ws, need = self._workspace(d, dev)
            q = th.empty(B, nt, self.n_agents, self.n_actions, dtype=th.float32, device=dev)
            _lib.check(_lib.lib().pmb_coma_critic_fwd(C.byref(d), C.byref(pb), _lib.ptr(flat),
                                                      t0, nt, _lib.ptr(q), _lib.ptr(ws), need, _lib.stream_ptr(dev)),
                       "pmb_coma_critic_fwd")
        return q


class CriticStep(th.autograd.Function):
    """COMACritic.forward over batch timesteps t0 .. t0 + nt - 1 as one autograd node: pmb_coma_critic_step_fwd (the same
    q bits as pmb_coma_critic_fwd) keeps the hidden activations x1, x2 [B * nt * N][E]; the backward is
    pmb_coma_critic_step_bwd from the dense dq.  src = (pmb_batch, [tensors the batch points into], flat parameter block).
    Returns q [B, nt, N, A]; gradients flow to the parameters (CRITIC_KEYS order), as views of a fresh block per call.
    Everything the backward reads is a saved tensor, so it is freed with the graph's buffers after the backward."""

    @staticmethod
    def forward(ctx, critic, dims, src, t0, nt, *params):
        batch, tensors, flat = src
        dev = flat.device
        B, N, A, E = dims.B, dims.N, dims.A, dims.E
        q = th.empty(B, nt, N, A, dtype=th.float32, device=dev)
        x1 = th.empty(B * nt * N, E, dtype=th.float32, device=dev)
        x2 = th.empty_like(x1)
        ws, need = critic._workspace(dims, dev)
        _lib.check(_lib.lib().pmb_coma_critic_step_fwd(C.byref(dims), C.byref(batch), _lib.ptr(flat), t0, nt, _lib.ptr(q),
                                                       _lib.ptr(x1), _lib.ptr(x2), _lib.ptr(ws), need, _lib.stream_ptr(dev)),
                   "pmb_coma_critic_step_fwd")
        # the parameters too: an in-place update before the backward raises
        ctx.save_for_backward(x1, x2, *tensors, *params)
        ctx.set_materialize_grads(False)
        ctx.step = (dims, batch, t0, nt, flat)
        return q

    @staticmethod
    def backward(ctx, dq):
        _lib.no_double_backward("COMACritic")
        dims, batch, t0, nt, flat = ctx.step
        saved = ctx.saved_tensors                             # also keeps alive (and version-checks) what `batch` points into
        params = saved[-len(CRITIC_KEYS):]
        if dq is None:
            return (None,) * (5 + len(params))
        x1, x2, dev = saved[0], saved[1], saved[0].device
        dq = dq.to(th.float32).contiguous()
        g = th.empty(sum(p.numel() for p in params), dtype=th.float32, device=dev)
        L = _lib.lib()
        nbytes = L.pmb_coma_critic_step_bwd_workspace_bytes(C.byref(dims), nt)
        scratch = th.empty(max(nbytes, 1), dtype=th.uint8, device=dev)
        _lib.check(L.pmb_coma_critic_step_bwd(C.byref(dims), C.byref(batch), _lib.ptr(flat), t0, nt, _lib.ptr(dq),
                                              _lib.ptr(x1), _lib.ptr(x2), _lib.ptr(g), _lib.ptr(scratch), nbytes,
                                              _lib.stream_ptr(dev)),
                   "pmb_coma_critic_step_bwd")
        grads, off = [], 0
        for p, need in zip(params, ctx.needs_input_grad[5:]):
            grads.append(g[off:off + p.numel()].view(p.shape) if need else None)
            off += p.numel()
        return (None,) * 5 + tuple(grads)
