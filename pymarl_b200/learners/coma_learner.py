"""COMALearner: counterfactual multi-agent policy gradients (reference: learners/coma_learner.py:9-184).

train(batch, t_env, episode_num) issues ONE C-ABI call (pmb_coma_train_step) for everything the reference does in Python:
the target critic over all timesteps, td-lambda targets, one critic optimiser step per timestep (backwards in time,
skipped where nothing is unmasked), the agent unroll, the policy head (masked softmax + epsilon floor + renormalisation),
the COMA loss, BPTT with the dense policy gradient and the agent's clip + RMSprop.  fp32 (CUDA-core) tier.  The host
reads the per-step statistics back once per call (the reference syncs ~5 times per timestep), counts the critic steps
that ran and does the hard target-critic sync.  Checkpoint files as in the reference: agent.th, critic.th, agent_opt.th,
critic_opt.th.
"""
import copy
import ctypes as C

import torch as th

from .. import _lib, flat as _flat
from ..modules.critics.coma import COMACritic, CRITIC_KEYS
from .q_learner import FusedRMSprop


class COMALearner:
    def __init__(self, mac, scheme, logger, args):
        self.args = args
        self.n_agents = args.n_agents
        self.n_actions = args.n_actions
        self.mac = mac
        self.logger = logger

        self.last_target_update_step = 0
        self.critic_training_steps = 0
        self.log_stats_t = -self.args.learner_log_interval - 1

        self.critic = COMACritic(scheme, args)
        self.target_critic = copy.deepcopy(self.critic)

        self.agent_params = list(mac.parameters())
        self.critic_params = list(self.critic.parameters())
        self.params = self.agent_params + self.critic_params

        self.agent_optimiser = FusedRMSprop(self.agent_params, lr=args.lr, alpha=args.optim_alpha, eps=args.optim_eps)
        self.critic_optimiser = FusedRMSprop(self.critic_params, lr=args.critic_lr, alpha=args.optim_alpha, eps=args.optim_eps)
        self._flat = None
        self._ws = None
        self._stats = None
        self._graphs = {}
        self.last_stats = None

    # ---- flat storage: agent [p | g | sq] in the Q-learner's agent layout, critic in state_dict order ---------------
    def _ensure_flat(self):
        agent = self.mac.agent
        _lib.require_cuda(agent.fc1.weight, "learner parameters (call learner.cuda())")
        dev = agent.fc1.weight.device
        a = self.args
        d_in = agent.d_in
        O = d_in - (a.n_actions if a.obs_last_action else 0) - (a.n_agents if a.obs_agent_id else 0)
        dims = _lib.make_dims(B=1, T=2, N=a.n_agents, O=O, S=1, A=a.n_actions, H=a.rnn_hidden_dim, E=1,
                              obs_last_action=a.obs_last_action, obs_agent_id=a.obs_agent_id, mixer=None)
        layout = _lib.flat_layout(dims)
        f = self._flat
        ok = f is not None and f["ap"].device == dev and _flat.block_ptr(agent, "agent", layout) == f["ap"].data_ptr() \
            and _flat.is_bound_in_order(self.critic, CRITIC_KEYS, f["cp"]) \
            and _flat.is_bound_in_order(self.target_critic, CRITIC_KEYS, f["tp"])
        if ok:
            return f
        na = layout.n_agent
        nc = sum(p.numel() for p in self.critic_params)
        z = lambda n: th.zeros(n, dtype=th.float32, device=dev)
        new = dict(ap=z(na), ag=z(na), asq=z(na), cp=z(nc), cg=z(nc), csq=z(nc), tp=z(nc), layout=layout, O=O)
        _flat.bind(new["ap"], layout, agent, "agent", grad=new["ag"])
        _flat.bind_in_order(self.critic, CRITIC_KEYS, new["cp"], grad=new["cg"])
        _flat.bind_in_order(self.target_critic, CRITIC_KEYS, new["tp"])
        for opt, params, flat_p, flat_sq in ((self.agent_optimiser, self.agent_params, new["ap"], new["asq"]),
                                             (self.critic_optimiser, self.critic_params, new["cp"], new["csq"])):
            views = []
            for p, old in zip(params, opt.square_avg):
                off = (p.data_ptr() - flat_p.data_ptr()) // 4
                v = flat_sq[off:off + p.numel()].view(p.shape)
                v.copy_(old.to(dev))
                views.append(v)
            opt.square_avg = views
        self._flat = new
        self._graphs = {}
        return new

    def train(self, batch, t_env: int, episode_num: int):
        if getattr(batch, "host_ids", None) is not None:
            raise TypeError("COMALearner does not take zero-copy samples of a host replay buffer; "
                            "set buffer.zero_copy = False for COMA")
        a = self.args
        f = self._ensure_flat()
        dev = f["ap"].device
        keep = []
        fields = {}
        for k in ("obs", "state", "actions", "avail_actions", "reward", "terminated", "filled"):
            t = batch[k]
            fields[k] = t if t.is_cuda else t.to(dev, non_blocking=True)
        B, T = fields["obs"].shape[0], fields["obs"].shape[1]
        S = 1
        for dim in fields["state"].shape[2:]:
            S *= int(dim)
        dims = _lib.make_dims(B=B, T=T, N=a.n_agents, O=f["O"], S=S, A=a.n_actions, H=a.rnn_hidden_dim,
                              E=COMACritic.HIDDEN, obs_last_action=a.obs_last_action, obs_agent_id=a.obs_agent_id, mixer=None)
        pb = _lib.make_batch(fields, need_state=True, keep=keep)
        L = _lib.lib()
        need = L.pmb_coma_workspace_bytes(C.byref(dims))
        if need < 0:
            _lib.check(1, "pmb_coma_workspace_bytes")
        if self._ws is None or self._ws.numel() < need or self._ws.device != dev:
            self._ws = None
            self._ws = th.empty(need, dtype=th.uint8, device=dev)
        n_rows = T                                          # (T-1) critic rows + 1 agent row
        if self._stats is None or self._stats.numel() < n_rows * _lib.STATS_LEN or self._stats.device != dev:
            self._stats = th.zeros(n_rows * _lib.STATS_LEN, dtype=th.float64, device=dev)
        ao, co = self.agent_optimiser.defaults, self.critic_optimiser.defaults
        epsilon = float(getattr(self.mac.action_selector, "epsilon", 0.0))
        hp = _lib.ComaHParams(a.gamma, a.td_lambda, ao["lr"], co["lr"], ao["alpha"], ao["eps"], a.grad_norm_clip, epsilon)
        def launch():
            _lib.check(L.pmb_coma_train_step(C.byref(dims), C.byref(pb), C.byref(hp), _lib.ptr(f["ap"]), _lib.ptr(f["ag"]),
                                             _lib.ptr(f["asq"]), _lib.ptr(f["cp"]), _lib.ptr(f["cg"]), _lib.ptr(f["csq"]),
                                             _lib.ptr(f["tp"]), _lib.ptr(self._ws), need, _lib.ptr(self._stats),
                                             _lib.stream_ptr(dev)), "pmb_coma_train_step")
        if getattr(a, "cuda_graph", False):
            # ~14 launches per timestep (one critic optimiser step each) + the agent pass: replay them as ONE graph, keyed
            # on everything the launches bake in (see QLearner._run_graphed); first sight eager, second captures
            key = (tuple(getattr(dims, k) for k, _ in dims._fields_), tuple(getattr(pb, k) for k, _ in pb._fields_),
                   tuple(getattr(hp, k) for k, _ in hp._fields_), f["ap"].data_ptr(), f["cp"].data_ptr(), self._ws.data_ptr(),
                   self._stats.data_ptr())
            entry = self._graphs.get(key)
            if entry is None:
                if len(self._graphs) >= 16:
                    self._graphs.pop(next(iter(self._graphs)))
                self._graphs[key] = "seen"
                launch()
            else:
                if entry == "seen":
                    g = th.cuda.CUDAGraph()
                    th.cuda.synchronize(dev)
                    with th.cuda.graph(g):
                        launch()
                    entry = self._graphs[key] = (g, list(keep))
                entry[0].replay()
        else:
            launch()
        if hasattr(self.mac, "params_changed"):
            self.mac.params_changed()
        self._last_dims = dims
        st = self._stats[:n_rows * _lib.STATS_LEN].view(n_rows, _lib.STATS_LEN).cpu()       # the one D2H sync of the step
        self.last_stats = st
        crit, ag = st[:T - 1], st[T - 1]
        ran = crit[:, 0] > 0                                 # `if mask_t.sum() == 0: continue` (coma_learner.py:120-121)
        n_ran = int(ran.sum())
        self.critic_training_steps += n_ran
        self.critic_optimiser.step_count += n_ran
        self.agent_optimiser.step_count += 1

        if (self.critic_training_steps - self.last_target_update_step) / a.target_update_interval >= 1.0:
            self._update_targets()
            self.last_target_update_step = self.critic_training_steps

        if t_env - self.log_stats_t >= a.learner_log_interval:
            c = crit[ran]
            ts_logged = max(1, n_ran)
            m = c[:, 0]
            self.logger.log_stat("critic_loss", float((c[:, 1] / m).sum()) / ts_logged, t_env)
            self.logger.log_stat("critic_grad_norm", float(c[:, 5].sum()) / ts_logged, t_env)
            self.logger.log_stat("td_error_abs", float((c[:, 2] / m).sum()) / ts_logged, t_env)
            self.logger.log_stat("q_taken_mean", float((c[:, 3] / m).sum()) / ts_logged, t_env)
            self.logger.log_stat("target_mean", float((c[:, 4] / m).sum()) / ts_logged, t_env)
            msum = float(ag[0])
            self.logger.log_stat("advantage_mean", float(ag[2]) / msum, t_env)
            self.logger.log_stat("coma_loss", -float(ag[1]) / msum, t_env)
            self.logger.log_stat("agent_grad_norm", float(ag[5]), t_env)
            self.logger.log_stat("pi_max", float(ag[3]) / msum, t_env)
            self.log_stats_t = t_env

    def workspace_views(self):
        """q_vals [B, T-1, N, A], td-lambda targets [B, T-1, N], pi and logits [T-1, B*N, A] of the latest step (tests)."""
        d = self._last_dims
        ptrs = [C.c_void_p() for _ in range(4)]
        _lib.check(_lib.lib().pmb_coma_workspace_views(C.byref(d), _lib.ptr(self._ws), *[C.byref(p) for p in ptrs]),
                   "pmb_coma_workspace_views")
        base, f32 = self._ws.data_ptr(), self._ws.view(th.float32)
        B, T, N, A = d.B, d.T, d.N, d.A
        shapes = [(B, T - 1, N, A), (B, T - 1, N), (T - 1, B * N, A), (T - 1, B * N, A)]
        out = []
        for p, shp in zip(ptrs, shapes):
            n = 1
            for s_ in shp:
                n *= s_
            off = (p.value - base) // 4
            out.append(f32[off:off + n].view(shp))
        return dict(q_vals=out[0], targets=out[1], pi=out[2], logits=out[3])

    def _update_targets(self):
        self.target_critic.load_state_dict(self.critic.state_dict())
        self.logger.console_logger.info("Updated target network")

    def cuda(self):
        self.mac.cuda()
        self.critic.cuda()
        self.target_critic.cuda()
        self._ensure_flat()

    def save_models(self, path):
        self.mac.save_models(path)
        th.save(self.critic.state_dict(), "{}/critic.th".format(path))
        th.save(self.agent_optimiser.state_dict(), "{}/agent_opt.th".format(path))
        th.save(self.critic_optimiser.state_dict(), "{}/critic_opt.th".format(path))

    def load_models(self, path):
        self.mac.load_models(path)
        self.critic.load_state_dict(th.load("{}/critic.th".format(path), map_location=lambda storage, loc: storage))
        # Like the reference (coma_learner.py:178-180): the target critic takes the loaded critic
        self.target_critic.load_state_dict(self.critic.state_dict())
        self.agent_optimiser.load_state_dict(th.load("{}/agent_opt.th".format(path), map_location=lambda storage, loc: storage))
        self.critic_optimiser.load_state_dict(th.load("{}/critic_opt.th".format(path), map_location=lambda storage, loc: storage))
