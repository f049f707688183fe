"""QMIX monotonic mixing network (reference: modules/mixers/qmix.py:7-47).

Parameters keep the reference names (hyper_w_1, hyper_w_final, hyper_b_1, V.0, V.2);
forward() runs pmb_mixer_fwd: one GEMM for the four state hypernets + a fused
abs / ELU / dot-product mixing kernel.

By default the module is inference only (the built-in learners own the backward).  With ``args.autograd_modules = True``
and grad mode on, forward() is one autograd node (QMixStep): pmb_mixer_bwd gives the gradients of the ten parameters
and of agent_qs (none flows into the states)."""
import ctypes as C

import numpy as np
import torch as th
import torch.nn as nn

from ... import _lib, flat as _flat


class QMixer(nn.Module):
    def __init__(self, args):
        super().__init__()
        self.args = args
        self.n_agents = args.n_agents
        self.state_dim = int(np.prod(args.state_shape))
        self.embed_dim = args.mixing_embed_dim
        self.hyper_w_1 = nn.Linear(self.state_dim, self.embed_dim * self.n_agents)
        self.hyper_w_final = nn.Linear(self.state_dim, self.embed_dim)
        self.hyper_b_1 = nn.Linear(self.state_dim, self.embed_dim)
        self.V = nn.Sequential(nn.Linear(self.state_dim, self.embed_dim), nn.ReLU(), nn.Linear(self.embed_dim, 1))

    def forward(self, agent_qs, states):
        """agent_qs [B, T', N], states [B, T', S] -> q_tot [B, T', 1]."""
        _lib.require_cuda(agent_qs, "agent_qs")
        if _lib.autograd_mode(self.args):
            if states.requires_grad:
                raise _lib.PmbError("QMixer: no gradient flows into the states (batch data); pass states.detach()")
            return QMixStep.apply(self, agent_qs, states, *self.parameters())
        with th.no_grad():
            return self._forward(agent_qs, states)[0]

    def _forward(self, agent_qs, states):
        """-> q_tot, and what the backward reads: dims, the flat block, the pmb_batch of the states, qs, st, raw."""
        bs, tp = agent_qs.shape[0], agent_qs.shape[1]
        qs = agent_qs.detach().to(th.float32).contiguous()
        st = states.detach().to(th.float32).reshape(bs, tp, self.state_dim).contiguous()
        # T = tp + 1 so that the kernel's [B, T-1] row space is exactly these rows
        dims = _lib.make_dims(B=bs, T=tp + 1, N=self.n_agents, O=1, S=self.state_dim, A=1, H=16,
                              E=self.embed_dim, mixer="qmix")
        flat_mixer = C.c_void_p(_flat.ensure_block(self, "mixer", dims))
        batch = _lib.Batch()
        batch.state = st.data_ptr()
        batch.state_sb = tp * self.state_dim
        raw = th.empty(bs * tp, (self.n_agents + 3) * self.embed_dim, dtype=th.float32, device=qs.device)
        q_tot = th.empty(bs, tp, 1, dtype=th.float32, device=qs.device)
        _lib.check(_lib.lib().pmb_mixer_fwd(C.byref(dims), C.byref(batch), flat_mixer,
                                            _lib.ptr(qs), 0, _lib.ptr(raw), _lib.ptr(q_tot),
                                            _lib.stream_ptr(qs.device)), "pmb_mixer_fwd")
        return q_tot, (dims, flat_mixer, batch, qs, st, raw)


class QMixStep(th.autograd.Function):
    """QMixer.forward as one autograd node: pmb_mixer_fwd keeps the hypernet outputs (raw), pmb_mixer_bwd maps
    g = dL/dq_tot to d agent_qs and the mixer's parameter gradients (a fresh block per call)."""

    @staticmethod
    def forward(ctx, mixer, agent_qs, states, *params):
        q_tot, (dims, flat_mixer, batch, qs, st, raw) = mixer._forward(agent_qs, states)
        ctx.save_for_backward(qs, st, raw, *params)
        ctx.mix = (mixer, dims, flat_mixer, batch, agent_qs.dtype)
        return q_tot

    @staticmethod
    def backward(ctx, g):
        _lib.no_double_backward("QMixer")
        qs, st, raw = ctx.saved_tensors[:3]
        mixer, dims, flat_mixer, batch, qs_dtype = ctx.mix
        dev = qs.device
        L = _lib.lib()
        layout = _lib.flat_layout(dims)
        g = g.to(th.float32).contiguous()
        raw = raw.clone()                                    # pmb_mixer_bwd overwrites it; backward may run again
        d_qs = th.empty_like(qs)
        gm = th.empty(_flat.block_numel(layout, "mixer"), dtype=th.float32, device=dev)
        nbytes = L.pmb_mixer_bwd_workspace_bytes(C.byref(dims))
        scratch = th.empty(nbytes, dtype=th.uint8, device=dev)
        _lib.check(L.pmb_mixer_bwd(C.byref(dims), C.byref(batch), flat_mixer, _lib.ptr(qs), _lib.ptr(raw), _lib.ptr(g),
                                   _lib.ptr(d_qs), _lib.ptr(gm), _lib.ptr(scratch), nbytes, _lib.stream_ptr(dev)),
                   "pmb_mixer_bwd")
        grads = [gv if need else None for gv, need in zip(_flat.grad_views(gm, layout, mixer, "mixer"), ctx.needs_input_grad[3:])]
        return (None, d_qs.to(qs_dtype) if ctx.needs_input_grad[1] else None, None) + tuple(grads)
