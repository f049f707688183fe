"""BasicMAC: shared-parameter multi-agent controller (reference: controllers/basic_controller.py:10-154).

forward() / select_actions() run one fused rollout step on the GPU (pmb_select_actions_step):
fc1 is evaluated without ever materialising the concatenated [obs | last-action one-hot |
agent-id one-hot] input (the one-hot blocks become column gathers of fc1.weight), followed by
the GRU cell, fc2, avail masking and epsilon-greedy selection.

Only the upstream configuration is implemented: agent "rnn", agent_output_type "q",
obs_decoder None, action_input_representation None (SURVEY.md section 2, row 3b).

Note on the last-action input: the reference reads ``actions_onehot[:, t-1]``; this package
reads ``actions[:, t-1]`` and ``filled[:, t-1]`` instead (the one-hot row is all-zero exactly
when the step was never written), so ``actions_onehot`` is never touched on the device.
"""
import ctypes as C

import torch as th

from .. import _lib, flat as _flat
from ..components.action_selectors import REGISTRY as action_REGISTRY
from ..modules.agents import REGISTRY as agent_REGISTRY


class BasicMAC:
    def __init__(self, scheme, groups, args):
        self.n_agents = args.n_agents
        self.args = args
        if getattr(args, "action_input_representation", None) is not None or getattr(args, "obs_decoder", None) is not None:
            raise NotImplementedError("pymarl_b200.BasicMAC implements the flat-observation RNN agent only")
        if getattr(args, "agent_output_type", "q") not in ("q", "pi_logits"):
            raise NotImplementedError("agent_output_type must be 'q' or 'pi_logits'")
        if getattr(args, "agent_output_type", "q") == "pi_logits" and not getattr(args, "mask_before_softmax", True):
            raise NotImplementedError("pi_logits is implemented with mask_before_softmax = True (the reference default)")
        input_shape = self._get_input_shape(scheme)
        self._build_agents(input_shape)
        self.agent_output_type = args.agent_output_type
        self.action_selector = action_REGISTRY[args.action_selector](args)
        self.hidden_states = None
        self._scratch = None
        self._weights_epoch = 0         # bumped by whoever rewrites the agent parameters behind torch's back (the learner's kernels)
        self._packed_key = None         # what the weight images in the rollout scratch were packed from
        self._dummies = None

    # ---- helpers ------------------------------------------------------------------------
    def _device(self):
        return self.agent.fc1.weight.device

    def _dims(self, ep_batch):
        a = self.args
        obs = ep_batch["obs"]
        return _lib.make_dims(B=ep_batch.batch_size, T=obs.shape[1], N=self.n_agents, O=obs.shape[-1], S=1,
                              A=a.n_actions, H=a.rnn_hidden_dim, E=1, obs_last_action=a.obs_last_action,
                              obs_agent_id=a.obs_agent_id, mixer=None, precision=getattr(a, "precision", "fp32"))

    def _step_batch(self, ep_batch, t, keep, dims):
        """pmb_batch with just the fields a rollout step reads.  When the runner keeps its
        batch on the host (reference behaviour, basic_controller.py:32,105,113) only the
        timesteps the step needs are copied, re-based so that the kernel's index t maps onto
        them.  bf16 obs and uint8 / bool avail stay as they are where the rollout kernels read them natively for ``dims``."""
        dev = self._device()
        fields = {}
        if ep_batch["obs"].is_cuda:
            for k in ("obs", "actions", "avail_actions", "filled"):
                fields[k] = ep_batch[k]
            t_local, T_local = t, ep_batch["obs"].shape[1]
        else:
            # actions / filled: steps t-1 and t (the last-action input); obs / avail_actions: step t only, presented
            # at the same local time index (they are 99 % of the bytes)
            lo = max(t - 1, 0)
            for k in ("actions", "filled"):
                fields[k] = _lib.h2d_time_slice(ep_batch[k], lo, t + 1, dev)
            for k in ("obs", "avail_actions"):
                fields[k] = _lib.h2d_time_slice(ep_batch[k], t, t + 1, dev, lead=t - lo)
            t_local, T_local = t - lo, t + 1 - lo
        # placeholders for the fields a rollout step never reads: created once per device (two tiny torch launches per
        # step were 4 % of the 16384-env step)
        if self._dummies is None or self._dummies[0].device != dev:
            zero = th.zeros(1, dtype=th.float32, device=dev)
            self._dummies = (zero, zero.to(th.uint8))
        zero, zero_u8 = self._dummies
        fields.update(state=zero, reward=zero, terminated=zero_u8)
        b = _lib.make_batch(fields, need_state=False, keep=keep, dims=dims, entry=_lib.ENTRY_SELECT_ACTIONS)
        return b, t_local, T_local

    def _run_step(self, ep_batch, t, epsilon=None, u=None, expo=None, seed=0, offset=0, want_actions=False, want_q=True):
        dev = self._device()
        _lib.require_cuda(self.agent.fc1.weight, "agent parameters")
        keep = []
        dims = self._dims(ep_batch)
        batch, t_local, T_local = self._step_batch(ep_batch, t, keep, dims)
        dims.T = T_local
        B, N, A, H = dims.B, dims.N, dims.A, dims.H
        flat = C.c_void_p(_flat.ensure_block(self.agent, "agent", dims))
        hs = self.hidden_states
        if hs is None:
            raise RuntimeError("call init_hidden(batch_size) before forward/select_actions")
        if (not hs.is_cuda) or hs.dtype != th.float32 or not hs.is_contiguous() or hs.numel() != B * N * H \
                or hs.data_ptr() % 16 != 0:
            hs = hs.expand(B, N, H).to(device=dev, dtype=th.float32).contiguous() if hs.dim() == 3 \
                else hs.reshape(-1, H).expand(B * N, H).to(device=dev, dtype=th.float32).contiguous()
        hs = hs.view(B * N, H)
        need = _lib.lib().pmb_select_actions_workspace_bytes(C.byref(dims))
        if self._scratch is None or self._scratch.numel() < need or self._scratch.device != dev:
            self._scratch = th.empty(need, dtype=th.uint8, device=dev)
        # packed weight images live in the scratch between steps: re-pack only when the parameters (or the scratch) changed
        key = (self._scratch.data_ptr(), flat.value, self._weights_epoch, dims.B, dims.O,
               tuple(p._version for p in self.agent.parameters()))
        dims.reserved = 1 if key == self._packed_key else 0
        self._packed_key = key
        q = th.empty(B, N, A, dtype=th.float32, device=dev) if (want_q or not want_actions) else None
        actions = th.empty(B, N, dtype=th.int64, device=dev) if want_actions else None
        _lib.check(_lib.lib().pmb_select_actions_step(
            C.byref(dims), C.byref(batch), t_local, flat, _lib.ptr(hs), C.c_float(epsilon or 0.0), _lib.ptr(u),
            _lib.ptr(expo), seed, offset, _lib.ptr(actions), _lib.ptr(q), _lib.ptr(self._scratch), need,
            _lib.stream_ptr(dev)), "pmb_select_actions_step")
        self.hidden_states = hs                   # [B*N, H], like the reference after the first step
        return q, actions

    # ---- reference surface ----------------------------------------------------------------
    def select_actions(self, ep_batch, t_ep, t_env, bs=slice(None), test_mode=False):
        """One agent step for ALL envs (terminated ones keep stepping their hidden state,
        basic_controller.py:33,49), then epsilon-greedy on the rows `bs` (:34-37)."""
        sel = self.action_selector
        full = isinstance(bs, slice) and bs == slice(None)
        if self.agent_output_type == "pi_logits":
            probs = self.forward(ep_batch, t_ep, test_mode=test_mode)
            avail = ep_batch["avail_actions"][:, t_ep]
            return sel.select_action(probs[bs].to(self._device()), avail[bs].to(self._device()), t_env, test_mode=test_mode)
        if full and sel.rng != "torch":
            sel.epsilon = 0.0 if test_mode else sel.schedule.eval(t_env)
            seed, offset = sel.next_philox()
            _, actions = self._run_step(ep_batch, t_ep, epsilon=sel.epsilon, seed=seed, offset=offset,
                                        want_actions=True, want_q=False)
            return actions
        q, _ = self._run_step(ep_batch, t_ep)
        avail = ep_batch["avail_actions"][:, t_ep]
        return sel.select_action(q[bs], avail[bs].to(q.device), t_env, test_mode=test_mode)

    def forward(self, ep_batch, t, test_mode=False):
        q, _ = self._run_step(ep_batch, t)
        if self.agent_output_type == "pi_logits":
            # basic_controller.py:55-71: masked softmax, epsilon floor over the available actions, unavailable -> 0
            avail = ep_batch["avail_actions"][:, t].to(device=q.device, dtype=th.int32).contiguous()
            probs = th.empty_like(q)
            rows, A = q.shape[0] * q.shape[1], q.shape[2]
            _lib.check(_lib.lib().pmb_policy_head(rows, A, C.c_float(float(self.action_selector.epsilon)), int(bool(test_mode)),
                                                  _lib.ptr(q), _lib.ptr(avail), _lib.ptr(probs), _lib.stream_ptr(q.device)),
                       "pmb_policy_head")
            q = probs
        return q.view(ep_batch.batch_size, self.n_agents, -1).to(ep_batch.device)

    def init_hidden(self, batch_size):
        self.hidden_states = self.agent.init_hidden().unsqueeze(0).expand(batch_size, self.n_agents, -1)

    def parameters(self):
        return self.agent.parameters()

    def params_changed(self):
        """Tell the controller that the agent parameters were rewritten in place by a kernel (QLearner.train does)."""
        self._weights_epoch += 1

    def load_state(self, other_mac):
        self.agent.load_state_dict(other_mac.agent.state_dict())
        self.params_changed()

    def cuda(self):
        self.agent.cuda()
        self.params_changed()

    def save_models(self, path):
        th.save(self.agent.state_dict(), "{}/agent.th".format(path))

    def load_models(self, path):
        self.agent.load_state_dict(th.load("{}/agent.th".format(path), map_location=lambda storage, loc: storage))
        self.params_changed()

    def _build_agents(self, input_shape):
        self.agent = agent_REGISTRY[self.args.agent](input_shape, self.args)

    def _get_input_shape(self, scheme):
        """D_in = obs + n_actions (obs_last_action) + n_agents (obs_agent_id)
        (basic_controller.py:137-154; also normalises int vshapes to tuples like the reference)."""
        from collections import OrderedDict
        for k in ("obs", "actions_onehot"):
            if k in scheme and isinstance(scheme[k]["vshape"], int):
                scheme[k]["vshape"] = (scheme[k]["vshape"],)
        obs_dim = scheme["obs"]["vshape"][0]
        d_in = obs_dim
        if self.args.obs_last_action:
            d_in += scheme["actions_onehot"]["vshape"][0] if "actions_onehot" in scheme else self.args.n_actions
        if self.args.obs_agent_id:
            d_in += self.n_agents
        return OrderedDict([("1d", (d_in,))])
