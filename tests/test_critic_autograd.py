"""Autograd through COMACritic (args.autograd_modules): what an actor-critic learner of the user's own needs when it calls
critic(batch, t), builds a loss of q and calls loss.backward() (learners/coma_learner.py:96-148 is the pattern).

The referee is float64 torch autograd over the reference critic: three nn.Linear layers on the input built in torch
exactly as modules/critics/coma.py:29-50 builds it, from actions_onehot.  Gradients are compared as max-norm relative
errors per tensor.  A learner restating coma_learner.py:37-148 on this package's BasicMAC and COMACritic must reproduce
the reference COMALearner's recorded run (tests/golden/coma_tiny.npz) within the bounds the fused path meets.
"""
import copy

import numpy as np
import pytest
import torch as th
import torch.nn as nn
import torch.nn.functional as F

from golden_utils import Golden, rel_err
from pymarl_b200 import _lib, mac_REGISTRY
from pymarl_b200.modules.critics.coma import COMACritic, CRITIC_KEYS
from pymarl_b200.synthetic import SMAC_SHAPES, default_args, get_shape, make_scheme, numpy_episode_fields
from test_coma_gpu import COMA_KW, TOL, build_coma, state_np, target_chunks

gpu = pytest.mark.gpu


# ---- float64 referee ------------------------------------------------------------------------------------------------
class RefCritic(nn.Module):
    def __init__(self, D, A, E=128):
        super().__init__()
        self.fc1 = nn.Linear(D, E)
        self.fc2 = nn.Linear(E, E)
        self.fc3 = nn.Linear(E, A)

    def forward(self, inputs):                              # coma.py:22-27, pre-activations kept for the tie check
        z1 = self.fc1(inputs)
        z2 = self.fc2(F.relu(z1))
        return self.fc3(F.relu(z2)), z1, z2


def ref_critic_inputs(f, t, N, A):
    """coma.py:29-50 on float64 tensors f["state"] [B, T, S], f["obs"] [B, T, N, O], f["actions_onehot"] [B, T, N, A]."""
    state, obs, oh = f["state"], f["obs"], f["actions_onehot"]
    bs = obs.shape[0]
    max_t = obs.shape[1] if t is None else 1
    ts = slice(None) if t is None else slice(t, t + 1)
    inputs = [state[:, ts].unsqueeze(2).repeat(1, 1, N, 1), obs[:, ts]]
    actions = oh[:, ts].reshape(bs, max_t, 1, -1).repeat(1, 1, N, 1)
    agent_mask = (1 - th.eye(N, dtype=oh.dtype, device=oh.device)).view(-1, 1).repeat(1, A).view(N, -1)
    inputs.append(actions * agent_mask.unsqueeze(0).unsqueeze(0))
    if t == 0:
        inputs.append(th.zeros_like(oh[:, 0:1]).reshape(bs, max_t, 1, -1).repeat(1, 1, N, 1))
    elif isinstance(t, int):
        inputs.append(oh[:, t - 1:t].reshape(bs, max_t, 1, -1).repeat(1, 1, N, 1))
    else:
        last = th.cat([th.zeros_like(oh[:, 0:1]), oh[:, :-1]], dim=1)
        inputs.append(last.reshape(bs, max_t, 1, -1).repeat(1, 1, N, 1))
    inputs.append(th.eye(N, dtype=oh.dtype, device=oh.device).unsqueeze(0).unsqueeze(0).expand(bs, max_t, -1, -1))
    return th.cat([x.reshape(bs, max_t, N, -1) for x in inputs], dim=-1)


def critic_args(shape, **over):
    return default_args(shape, mixer=None, **dict(dict(autograd_modules=True, device="cuda"), **over))


def make_critic(shape, args, seed=0):
    th.manual_seed(seed)
    scheme, _ = make_scheme(shape)
    return COMACritic(scheme, args).cuda()


def episode(shape, B, T, seed):
    from cuda_utils import to_batch
    fields = numpy_episode_fields(shape, B, T, seed=seed, ragged=True)
    return fields, to_batch(shape, fields)


def test_critic_parameters_are_in_the_flat_layout_order():
    """CriticStep hands gradients back in parameters() order; the kernels write them in CRITIC_KEYS order."""
    shape = SMAC_SHAPES["3m"]
    scheme, _ = make_scheme(shape)
    critic = COMACritic(scheme, default_args(shape, mixer=None))
    assert [k for k, _ in critic.named_parameters()] == CRITIC_KEYS


# (shape, B, T): 27m_vs_30m at the reference's on-policy batch gives A > 32, a t = None pass in two chunks and, at a single
# step, 216 rows, more than one row slice of the weight gradients (see test_backward_is_deterministic...)
REF_SHAPES = {"3m": (5, 9), "2s3z": (6, 10), "MMM2": (4, 12), "27m_vs_30m": (8, 120)}


@gpu
@pytest.mark.parametrize("form", ["t0", "t_last", "all"])
@pytest.mark.parametrize("shape_key", list(REF_SHAPES))
def test_critic_forward_backward_matches_float64(shape_key, form):
    shape = get_shape(shape_key)
    B, T = REF_SHAPES[shape_key]
    N, A = shape.n_agents, shape.n_actions
    if shape_key == "27m_vs_30m":
        assert A > 32 and len(target_chunks(shape, B, T)) == 2
    t = {"t0": 0, "t_last": T - 1, "all": None}[form]
    args = critic_args(shape)
    critic = make_critic(shape, args, seed=len(shape_key))
    fields, batch = episode(shape, B, T, seed=3)
    assert (fields["filled"] == 0).any()                    # ragged: unfilled steps
    f64 = {k: th.from_numpy(fields[k]).double().cuda() for k in ("state", "obs", "actions_onehot")}
    inp = ref_critic_inputs(f64, t, N, A)
    ref = RefCritic(inp.shape[-1], A).double().cuda()
    ref.load_state_dict({k: v.detach().double() for k, v in critic.state_dict().items()})
    q_ref, z1, z2 = ref(inp)
    # Rows with a pre-activation within rounding of zero may take the other ReLU branch in fp32: they get no weight in
    # the loss, so either branch gives the same gradients.  Unfilled rows of an agent share one input, so they tie
    # together (1079 of 25920 rows at 27m_vs_30m t = None, a few or none elsewhere).
    tie = th.minimum(z1.abs().amin(-1), z2.abs().amin(-1)) < 1e-5
    w = th.from_numpy(np.random.default_rng(7).standard_normal(tuple(q_ref.shape))).cuda() * (~tie)[..., None]
    (q_ref * w).sum().backward()

    q = critic(batch, t)
    assert q.grad_fn is not None and q.shape == (B, 1 if t is not None else T, N, A)
    (q * w.float()).sum().backward()
    errs = {"q": rel_err(q.detach().cpu(), q_ref.detach().cpu())}
    refp = dict(ref.named_parameters())
    errs.update({k: rel_err(p.grad.cpu(), refp[k].grad.cpu()) for k, p in critic.named_parameters()})
    print(shape_key, form, int(tie.sum()), {k: "%.1e" % v for k, v in errs.items()})
    assert all(e < 1e-5 for e in errs.values()), errs


# ---- the reference algorithm as a custom learner ----------------------------------------------------------------------
def build_td_lambda_targets(rewards, terminated, mask, target_qs, n_agents, gamma, td_lambda):   # utils/rl_utils.py:4-15
    ret = target_qs.new_zeros(*target_qs.shape)
    ret[:, -1] = target_qs[:, -1] * (1 - th.sum(terminated, dim=1))
    for t in range(ret.shape[1] - 2, -1, -1):
        ret[:, t] = td_lambda * gamma * ret[:, t + 1] + mask[:, t] \
            * (rewards[:, t] + (1 - td_lambda) * gamma * target_qs[:, t + 1] * (1 - terminated[:, t]))
    return ret[:, 0:-1]


class CustomCOMALearner:
    """learners/coma_learner.py:9-148 restated on any MAC and critic: torch RMSprop and clip_grad_norm_, one critic step
    per timestep backwards in time, the actor loss through mac.forward with pi_logits.  stats: what the reference logs."""

    def __init__(self, mac, critic, args):
        self.mac, self.critic, self.args = mac, critic, args
        self.n_agents, self.n_actions = args.n_agents, args.n_actions
        self.target_critic = copy.deepcopy(critic)
        self.agent_params = list(mac.parameters())
        self.critic_params = list(critic.parameters())
        self.agent_optimiser = th.optim.RMSprop(params=self.agent_params, lr=args.lr, alpha=args.optim_alpha, eps=args.optim_eps)
        self.critic_optimiser = th.optim.RMSprop(params=self.critic_params, lr=args.critic_lr, alpha=args.optim_alpha,
                                                 eps=args.optim_eps)
        self.critic_training_steps = 0
        self.last_target_update_step = 0
        self.stats = {}

    def train(self, batch):
        max_t = batch.max_seq_length
        rewards = batch["reward"][:, :-1]
        actions = batch["actions"][:, :]
        terminated = batch["terminated"][:, :-1].float()
        mask = batch["filled"][:, :-1].float()
        mask[:, 1:] = mask[:, 1:] * (1 - terminated[:, :-1])
        avail_actions = batch["avail_actions"][:, :-1]
        critic_mask = mask.clone()
        mask = mask.repeat(1, 1, self.n_agents).view(-1)

        q_vals, log = self._train_critic(batch, rewards, terminated, actions, critic_mask)
        actions = actions[:, :-1]
        mac_out = []
        self.mac.init_hidden(batch.batch_size)
        for t in range(max_t - 1):
            mac_out.append(self.mac.forward(batch, t=t))
        mac_out = th.stack(mac_out, dim=1)
        mac_out[avail_actions == 0] = 0
        mac_out = mac_out / mac_out.sum(dim=-1, keepdim=True)
        mac_out[avail_actions == 0] = 0

        q_vals = q_vals.reshape(-1, self.n_actions)
        pi = mac_out.view(-1, self.n_actions)
        baseline = (pi * q_vals).sum(-1).detach()
        q_taken = th.gather(q_vals, dim=1, index=actions.reshape(-1, 1)).squeeze(1)
        pi_taken = th.gather(pi, dim=1, index=actions.reshape(-1, 1)).squeeze(1)
        pi_taken[mask == 0] = 1.0
        log_pi_taken = th.log(pi_taken)
        advantages = (q_taken - baseline).detach()
        coma_loss = -((advantages * log_pi_taken) * mask).sum() / mask.sum()

        self.agent_optimiser.zero_grad()
        coma_loss.backward()
        grad_norm = th.nn.utils.clip_grad_norm_(self.agent_params, self.args.grad_norm_clip)
        self.agent_optimiser.step()

        if (self.critic_training_steps - self.last_target_update_step) / self.args.target_update_interval >= 1.0:
            self.target_critic.load_state_dict(self.critic.state_dict())
            self.last_target_update_step = self.critic_training_steps

        n = len(log["critic_loss"])
        self.stats = {k: sum(v) / n for k, v in log.items()}
        self.stats.update(advantage_mean=(advantages * mask).sum().item() / mask.sum().item(), coma_loss=coma_loss.item(),
                          agent_grad_norm=float(grad_norm),
                          pi_max=(pi.max(dim=1)[0] * mask).sum().item() / mask.sum().item())

    def _train_critic(self, batch, rewards, terminated, actions, mask):
        with th.no_grad():
            target_q_vals = self.target_critic(batch)[:, :]
        targets_taken = th.gather(target_q_vals, dim=3, index=actions).squeeze(3)
        targets = build_td_lambda_targets(rewards, terminated, mask, targets_taken, self.n_agents, self.args.gamma,
                                          self.args.td_lambda)
        q_vals = th.zeros_like(target_q_vals)[:, :-1]
        log = {k: [] for k in ("critic_loss", "critic_grad_norm", "td_error_abs", "target_mean", "q_taken_mean")}
        for t in reversed(range(rewards.size(1))):
            mask_t = mask[:, t].expand(-1, self.n_agents)
            if mask_t.sum() == 0:
                continue
            q_t = self.critic(batch, t)
            q_vals[:, t] = q_t.detach().view(-1, self.n_agents, self.n_actions)
            q_taken = th.gather(q_t, dim=3, index=actions[:, t:t + 1]).squeeze(3).squeeze(1)
            targets_t = targets[:, t]
            masked_td_error = (q_taken - targets_t.detach()) * mask_t
            loss = (masked_td_error ** 2).sum() / mask_t.sum()
            self.critic_optimiser.zero_grad()
            loss.backward()
            grad_norm = th.nn.utils.clip_grad_norm_(self.critic_params, self.args.grad_norm_clip)
            self.critic_optimiser.step()
            self.critic_training_steps += 1
            mask_elems = mask_t.sum().item()
            log["critic_loss"].append(loss.item())
            log["critic_grad_norm"].append(float(grad_norm))
            log["td_error_abs"].append(masked_td_error.abs().sum().item() / mask_elems)
            log["q_taken_mean"].append((q_taken * mask_t).sum().item() / mask_elems)
            log["target_mean"].append((targets_t * mask_t).sum().item() / mask_elems)
        return q_vals, log


def package_learner(shape, args, agent=None, critic=None, target_critic=None):
    """CustomCOMALearner on this package's BasicMAC and COMACritic."""
    scheme, groups = make_scheme(shape)
    scheme["actions_onehot"] = {"vshape": (shape.n_actions,), "dtype": th.float32, "group": "agents"}
    mac = mac_REGISTRY[args.mac](copy.deepcopy(scheme), groups, args)
    mac.cuda()
    crit = COMACritic(scheme, args).cuda()
    ld = lambda m, p: m.load_state_dict({k: th.from_numpy(np.asarray(v, np.float32)) for k, v in p.items()}) if p else None
    ld(mac.agent, agent)
    ld(crit, critic)
    learner = CustomCOMALearner(mac, crit, args)
    ld(learner.target_critic, target_critic)
    return learner


@gpu
def test_reference_learner_on_the_modules_matches_golden():
    """Bounds of test_coma_train_steps_match_reference_golden (the fused learner step on the same fixture)."""
    from cuda_utils import to_batch
    g = Golden("coma_tiny")
    args = default_args(g.shape, mixer=None, **dict(g.meta["over"], autograd_modules=True, device="cuda", use_cuda=True))
    learner = package_learner(g.shape, args, g.group("init/agent"), g.group("init/critic"), g.group("init/target_critic"))
    batch = to_batch(g.shape, g.batch_fields())
    learner.mac.action_selector.epsilon = float(g["epsilon"])
    for step in range(g.meta["n_steps"]):
        learner.train(batch)
        for k in ("critic_loss", "critic_grad_norm", "td_error_abs", "q_taken_mean", "target_mean", "advantage_mean",
                  "coma_loss", "agent_grad_norm", "pi_max"):
            r = float(g["step%d/stat/%s" % (step, k)])
            assert abs(learner.stats[k] - r) <= 3 * TOL * max(1.0, abs(r)), (step, k, learner.stats[k], r)
        for tag, mod in (("agent", learner.mac.agent), ("critic", learner.critic), ("target_critic", learner.target_critic)):
            for k, v in g.group("step%d/%s" % (step, tag)).items():
                assert rel_err(state_np(mod)[k], v) < 5 * TOL, (step, tag, k)
        assert learner.critic_training_steps == int(g["step%d/critic_training_steps" % step])
        for tag, opt, params in (("agent", learner.agent_optimiser, learner.agent_params),
                                 ("critic", learner.critic_optimiser, learner.critic_params)):
            sq = np.concatenate([opt.state[p]["square_avg"].cpu().numpy().ravel() for p in params])
            assert rel_err(sq, g["step%d/sq/%s" % (step, tag)]) < 1e-4, (step, tag)


# ---- bits, bookkeeping, determinism, launches, double backward --------------------------------------------------------
@gpu
@pytest.mark.parametrize("shape_key, B, T", [("2s3z", 6, 10), ("27m_vs_30m", 8, 120)])
def test_key_on_and_off_give_the_same_q_bits(shape_key, B, T):
    shape = get_shape(shape_key)
    on = critic_args(shape)
    critic = make_critic(shape, on)
    _, batch = episode(shape, B, T, seed=4)
    for t in (None, 0, T // 2):
        q_on = critic(batch, t)
        assert q_on.grad_fn is not None
        critic.args = critic_args(shape, autograd_modules=False)
        q_off = critic(batch, t)
        critic.args = on
        with th.no_grad():
            q_ng = critic(batch, t)
        with th.inference_mode():
            q_inf = critic(batch, t)
        assert q_off.grad_fn is None and q_ng.grad_fn is None and not q_off.requires_grad
        assert th.equal(q_on.detach(), q_off) and th.equal(q_off, q_ng) and th.equal(q_off, q_inf), t


def _critic_loss(critic, batch, ts):
    out = 0
    for t in ts:
        q = critic(batch, t)
        w = th.linspace(-1, 1, q.shape[-1], device="cuda")
        out = out + (q * w).sum() * (1.0 if t is None else 1 + 0.1 * t)
    return out


@gpu
def test_gradients_accumulate_into_bound_views_and_after_set_to_none():
    """COMALearner points the critic's .grad at views of its flat gradient buffer: AccumulateGrad adds into them in place;
    with the grads set to None it creates fresh ones; a torch optimiser step is seen by the next forward."""
    shape = get_shape("2s3z")
    args = critic_args(shape)
    critic = make_critic(shape, args)
    _, batch = episode(shape, 6, 10, seed=5)
    ts = [None, 3, 0]
    params = list(critic.parameters())
    _critic_loss(critic, batch, ts).backward()
    g1 = [p.grad.clone() for p in params]

    learner, _ = build_coma(shape, critic_args(shape, **COMA_KW))
    lc = learner.critic
    lc.load_state_dict(critic.state_dict())
    flat_g = learner._flat["cg"]
    flat_g.fill_(0.5)
    for p in lc.parameters():
        assert p.grad is not None and flat_g.data_ptr() <= p.grad.data_ptr() < flat_g.data_ptr() + 4 * flat_g.numel()
    _critic_loss(lc, batch, ts).backward()
    for p, g in zip(lc.parameters(), g1):
        assert rel_err(p.grad.cpu(), (g + 0.5).cpu()) < 1e-6
        assert flat_g.data_ptr() <= p.grad.data_ptr() < flat_g.data_ptr() + 4 * flat_g.numel()

    for p in params:
        p.grad = None
    _critic_loss(critic, batch, ts).backward()
    _critic_loss(critic, batch, ts).backward()
    for p, g in zip(params, g1):
        assert rel_err(p.grad.cpu(), (2 * g).cpu()) < 1e-6

    opt = th.optim.SGD(params, lr=0.05)
    opt.step()
    opt.zero_grad(set_to_none=True)
    with th.no_grad():
        q_after = critic(batch, 2)
    fields = {k: batch[k][:, :].double() for k in ("state", "obs", "actions_onehot")}
    inp = ref_critic_inputs(fields, 2, shape.n_agents, shape.n_actions)
    ref = RefCritic(inp.shape[-1], shape.n_actions).double().cuda()
    ref.load_state_dict({k: v.detach().double() for k, v in critic.state_dict().items()})
    assert rel_err(q_after.cpu(), ref(inp)[0].detach().cpu()) < 1e-5


@gpu
@pytest.mark.parametrize("shape_key, B, launches", [("3m", 4, 2), ("27m_vs_30m", 8, 3)])
def test_backward_is_deterministic_and_within_the_launch_budget(shape_key, B, launches):
    """One step: 3m at B = 4 is 12 rows, one row slice (2 launches); 27m_vs_30m at B = 8 is 216 rows, two slices and the
    ordered reduction (3 launches).  Two backward passes over the same graph, and a fresh graph, give the same bits."""
    shape = get_shape(shape_key)
    critic = make_critic(shape, critic_args(shape))
    T = 12
    _, batch = episode(shape, B, T, seed=6)
    params = list(critic.parameters())
    L = _lib.lib()
    for ts in ([5], [None]):
        loss = _critic_loss(critic, batch, ts)
        th.cuda.synchronize()
        n0 = L.pmb_launch_count()
        g_a = th.autograd.grad(loss, params, retain_graph=True)
        n1 = L.pmb_launch_count()
        g_b = th.autograd.grad(loss, params)
        g_c = th.autograd.grad(_critic_loss(critic, batch, ts), params)
        if ts == [5]:
            assert n1 - n0 == launches, (n1 - n0)
        assert n1 - n0 <= 3
        for a, b, c in zip(g_a, g_b, g_c):
            assert th.equal(a, b) and th.equal(a, c)


@gpu
def test_double_backward_raises_a_clear_error():
    shape = get_shape("3m")
    critic = make_critic(shape, critic_args(shape))
    _, batch = episode(shape, 3, 5, seed=8)
    with pytest.raises(_lib.PmbError, match="double backward"):
        _critic_loss(critic, batch, [1]).backward(create_graph=True)
