"""VDN mixer: q_tot = sum over agents (reference: modules/mixers/vdn.py:5-10).

Parameter-free.  The learner's fused step never materialises this module's output (the VDN sum lives inside
pmb_qlearner_train_step); a standalone call runs the same kernel through pmb_mixer_fwd (VDN variant).  When grad mode
is on and agent_qs requires grad, the sum is th.sum, so the gradient reaches agent_qs (a user's learner calling
loss.backward())."""
import ctypes as C

import torch as th
import torch.nn as nn

from ... import _lib


class VDNMixer(nn.Module):
    def __init__(self):
        super().__init__()

    def forward(self, agent_qs, batch):
        """agent_qs [B, T', N] -> [B, T', 1]; the second argument (the states) is unused, as in the reference."""
        _lib.require_cuda(agent_qs, "agent_qs")
        if th.is_grad_enabled() and agent_qs.requires_grad:
            return th.sum(agent_qs, dim=2, keepdim=True)
        with th.no_grad():
            return self._forward(agent_qs)

    def _forward(self, agent_qs):
        bs, tp, n = agent_qs.shape
        qs = agent_qs.detach().to(th.float32).contiguous()
        dims = _lib.make_dims(B=bs, T=tp + 1, N=n, O=1, S=1, A=1, H=16, E=1, mixer="vdn")
        q_tot = th.empty(bs, tp, 1, dtype=th.float32, device=qs.device)
        _lib.check(_lib.lib().pmb_mixer_fwd(C.byref(dims), C.byref(_lib.Batch()), None, _lib.ptr(qs), 0, None,
                                            _lib.ptr(q_tot), _lib.stream_ptr(qs.device)), "pmb_mixer_fwd")
        return q_tot
