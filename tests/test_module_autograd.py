"""Autograd through RNNAgent, BasicMAC, QMixer and VDNMixer (args.autograd_modules): what a user's learner needs when it
unrolls mac.forward(batch, t), mixes, builds a loss and calls loss.backward().

The referee is float64 torch autograd on the CPU over a plain-torch restatement of the reference modules (nn.Linear /
nn.GRUCell as modules/agents/rnn_agent.py uses them, QMixer as modules/mixers/qmix.py:28-47 writes it).  Gradients are
compared as max-norm relative errors per tensor.  A custom learner restating learners/q_learner.py:37-103 on these
modules must give the gradient of the fused learner step (pmb_qlearner_train_step with skip_update = 1, the gradient of
sum((td * mask)^2)) once multiplied by sum(mask).
"""
import copy
import ctypes as C

import numpy as np
import pytest
import torch as th
import torch.nn as nn
import torch.nn.functional as F

from golden_utils import rel_err
from oracle import qlearner_oracle as orc
from pymarl_b200 import _lib, mac_REGISTRY
from pymarl_b200.modules.agents.rnn_agent import RNNAgent
from pymarl_b200.modules.mixers.qmix import QMixer
from pymarl_b200.modules.mixers.vdn import VDNMixer
from pymarl_b200.synthetic import SMAC_SHAPES, SmacShape, default_args, make_scheme, numpy_episode_fields


# ---- float64 referee ------------------------------------------------------------------------------------------------
class RefAgent(nn.Module):
    def __init__(self, d_in, H, A):
        super().__init__()
        self.fc1 = nn.Linear(d_in, H)
        self.rnn = nn.GRUCell(H, H)
        self.fc2 = nn.Linear(H, A)

    def forward(self, x, h):
        h = self.rnn(F.relu(self.fc1(x)), h)
        return self.fc2(h), h


class RefQMixer(nn.Module):
    def __init__(self, S, N, E):
        super().__init__()
        self.n_agents, self.state_dim, self.embed_dim = N, S, E
        self.hyper_w_1 = nn.Linear(S, E * N)
        self.hyper_w_final = nn.Linear(S, E)
        self.hyper_b_1 = nn.Linear(S, E)
        self.V = nn.Sequential(nn.Linear(S, E), nn.ReLU(), nn.Linear(E, 1))

    def forward(self, agent_qs, states):                  # qmix.py:28-47
        bs = agent_qs.size(0)
        states = states.reshape(-1, self.state_dim)
        agent_qs = agent_qs.view(-1, 1, self.n_agents)
        w1 = th.abs(self.hyper_w_1(states))
        b1 = self.hyper_b_1(states)
        w1 = w1.view(-1, self.n_agents, self.embed_dim)
        b1 = b1.view(-1, 1, self.embed_dim)
        hidden = F.elu(th.bmm(agent_qs, w1) + b1)
        w_final = th.abs(self.hyper_w_final(states)).view(-1, self.embed_dim, 1)
        v = self.V(states).view(-1, 1, 1)
        return (th.bmm(hidden, w_final) + v).view(bs, -1, 1)


def ref_of(module, ref):
    """float64 CPU copy of `module`'s parameters in the reference module `ref`."""
    ref.load_state_dict({k: v.detach().cpu().double() for k, v in module.state_dict().items()})
    return ref.double()


def ref_inputs(fields, t, N, A, last_action, agent_id):
    """basic_controller.py:100-135 from the numpy fields (last-action one-hot zero where step t-1 is not filled)."""
    obs = th.from_numpy(fields["obs"][:, t]).double()
    B = obs.shape[0]
    parts = [obs]
    if last_action:
        oh = th.zeros(B, N, A, dtype=th.float64)
        if t > 0:
            act = th.from_numpy(fields["actions"][:, t - 1, :, 0])
            oh.scatter_(2, act[..., None], 1.0)
            oh *= th.from_numpy(fields["filled"][:, t - 1, 0]).double()[:, None, None]
        parts.append(oh)
    if agent_id:
        parts.append(th.eye(N, dtype=th.float64).expand(B, N, N))
    return th.cat(parts, -1).reshape(B * N, -1)


def ref_policy(q, avail, eps, test_mode):
    off = avail == 0
    p = th.softmax(q.masked_fill(off, -1e10), dim=-1)
    if not test_mode:
        p = ((1.0 - eps) * p + eps / (~off).sum(-1, keepdim=True).double()).masked_fill(off, 0.0)
    return p


def grad_errs(named, ref_named):
    return {k: rel_err(p.grad.detach().cpu().numpy(), ref_named[k].grad.numpy()) for k, p in named}


def agent_args(shape, H=64, **over):
    return default_args(shape, **dict(dict(rnn_hidden_dim=H, autograd_modules=True, device="cuda"), **over))


def load_agent(agent, d_in, H, A, seed):
    params = orc.init_params(orc.agent_param_shapes(d_in, H, A), np.random.default_rng(seed))
    agent.load_state_dict({k: th.from_numpy(v) for k, v in params.items()})


# ---- host only --------------------------------------------------------------------------------------------------------
def test_autograd_mode_is_opt_in_and_follows_grad_mode():
    """No device call: the switch is off by default, and off under th.no_grad() / th.inference_mode()."""
    shape = SMAC_SHAPES["3m"]
    assert not _lib.autograd_mode(default_args(shape))
    on = default_args(shape, autograd_modules=True)
    assert _lib.autograd_mode(on)
    with th.no_grad():
        assert not _lib.autograd_mode(on)
    with th.inference_mode():
        assert not _lib.autograd_mode(on)


def test_cpu_inputs_still_have_no_cpu_path_with_the_key_on():
    shape = SMAC_SHAPES["3m"]
    args = default_args(shape, autograd_modules=True)
    N, A, H = shape.n_agents, shape.n_actions, args.rnn_hidden_dim
    agent = RNNAgent((shape.obs_dim,), args)
    with pytest.raises(_lib.PmbError, match="no CPU path"):
        agent(th.zeros(4, shape.obs_dim), th.zeros(4, H))
    with pytest.raises(_lib.PmbError, match="no CPU path"):
        QMixer(args)(th.zeros(2, 3, N, requires_grad=True), th.zeros(2, 3, shape.state_dim))
    with pytest.raises(_lib.PmbError, match="no CPU path"):
        VDNMixer()(th.zeros(2, 3, N, requires_grad=True), None)
    scheme, groups = make_scheme(shape)
    mac = mac_REGISTRY["basic_mac"](scheme, groups, args)
    fields = {k: th.from_numpy(v) for k, v in numpy_episode_fields(shape, 2, 4, seed=0).items()}
    mac.init_hidden(2)
    with pytest.raises(_lib.PmbError, match="no CPU path"):
        mac.forward(type("B", (), {"batch_size": 2, "device": "cpu", "__getitem__": lambda s, k: fields[k]})(), 0)


# ---- GPU: modules against the float64 referee -------------------------------------------------------------------------
@pytest.mark.gpu
def test_key_off_outputs_carry_no_graph_and_keep_their_bits():
    from cuda_utils import to_batch
    shape = SMAC_SHAPES["3m"]
    N, A = shape.n_agents, shape.n_actions
    for on in (False, True):
        th.manual_seed(0)
        args = default_args(shape, device="cuda", autograd_modules=on)
        d_in = shape.obs_dim + A + N
        agent = RNNAgent((d_in,), args).cuda()
        x, h = th.randn(12, d_in, device="cuda"), th.randn(12, args.rnn_hidden_dim, device="cuda")
        mixer = QMixer(args).cuda()
        qs, st = th.randn(4, 5, N, device="cuda"), th.randn(4, 5, shape.state_dim, device="cuda")
        scheme, groups = make_scheme(shape)
        mac = mac_REGISTRY["basic_mac"](scheme, groups, args)
        mac.agent.load_state_dict(agent.state_dict())
        mac.cuda()
        batch = to_batch(shape, {k: v for k, v in numpy_episode_fields(shape, 4, 6, seed=3).items() if k != "actions_onehot"})
        mac.init_hidden(4)
        if on:
            with th.no_grad():             # grad mode off: the inference kernels, whatever the key says
                outs = [agent(x, h)[0], agent(x, h)[1], mixer(qs, st), mac.forward(batch, 0), mac.forward(batch, 1)]
            ref = [o.clone() for o in outs_off]
            for a, b in zip(outs, ref):
                assert th.equal(a, b)
        else:
            outs_off = [agent(x, h)[0], agent(x, h)[1], mixer(qs, st), mac.forward(batch, 0), mac.forward(batch, 1)]
            assert not any(o.requires_grad for o in outs_off)
        acts = mac.select_actions(batch, t_ep=2, t_env=0)
        assert not acts.requires_grad and not mac.hidden_states.requires_grad


def _sm_count():
    sm, major, minor, smem = C.c_int32(), C.c_int32(), C.c_int32(), C.c_int64()
    _lib.check(_lib.lib().pmb_device_info(C.byref(sm), C.byref(major), C.byref(minor), C.byref(smem)), "pmb_device_info")
    return sm.value


# rows "wide": enough 64-row tiles to fill the machine twice, so pmb_agent_step_bwd runs its 64-row-tile kernel, and far
# more than 128 rows, so the weight gradients go through the row slices and their reduction
@pytest.mark.gpu
@pytest.mark.parametrize("H, rows", [(16, 45), (32, 45), (64, 45), (128, 45), (64, "wide"), (128, "wide")])
def test_rnn_agent_forward_backward_matches_float64(H, rows):
    shape = SmacShape("t", 5, 37, 20, 11, 10)
    args = agent_args(shape, H)
    rows = 2 * _sm_count() * 64 + 37 if rows == "wide" else rows
    d_in, A = shape.obs_dim, shape.n_actions
    agent = RNNAgent((d_in,), args).cuda()
    load_agent(agent, d_in, H, A, seed=H)
    ref = ref_of(agent, RefAgent(d_in, H, A))
    rng = np.random.default_rng(H + 1)
    x = rng.standard_normal((rows, d_in))
    h0 = 0.5 * rng.standard_normal((rows, H))
    wq, wh = rng.standard_normal((rows, A)), rng.standard_normal((rows, H))
    hd = th.tensor(h0, dtype=th.float32, device="cuda", requires_grad=True)
    q, h = agent(th.tensor(x, dtype=th.float32, device="cuda"), hd)
    assert q.requires_grad and h.requires_grad
    ((q * th.tensor(wq, device="cuda", dtype=th.float32)).sum() + (h * th.tensor(wh, device="cuda", dtype=th.float32)).sum()).backward()
    hr = th.tensor(h0, requires_grad=True)
    qr, hr_out = ref(th.tensor(x), hr)
    ((qr * th.tensor(wq)).sum() + (hr_out * th.tensor(wh)).sum()).backward()
    errs = {"q": rel_err(q.detach().cpu(), qr.detach()), "h": rel_err(h.detach().cpu(), hr_out.detach()),
            "dh0": rel_err(hd.grad.cpu(), hr.grad)}
    errs.update(grad_errs(agent.named_parameters(), dict(ref.named_parameters())))
    print(H, rows, {k: "%.1e" % v for k, v in errs.items()})
    assert all(e < 1e-5 for e in errs.values()), errs
    with pytest.raises(_lib.PmbError, match="agent inputs"):
        agent(th.zeros(rows, d_in, device="cuda", requires_grad=True), hd)


# id: (shape, overrides, B, T, batch layout).  B N > 128 rows ("sliced", "compact") sends the weight gradients of
# pmb_agent_step_bwd through the row slices and their reduction; the others run one slice.
MAC_CASES = {
    "sliced": ("2s3z", {}, 32, 12, "device"),
    "compact": ("2s3z", {}, 32, 12, "compact"),
    "q": ("3m", {}, 9, 12, "device"),
    "no_inputs": ("2s3z", dict(obs_last_action=False, obs_agent_id=False), 7, 12, "device"),
    "last_action_only_h32": ("3m", dict(obs_agent_id=False, rnn_hidden_dim=32), 9, 12, "device"),
    "host": ("2s3z", {}, 7, 12, "host"),
    "view": ("3m", {}, 9, 12, "view"),
    "pi_logits": ("3m", dict(agent_output_type="pi_logits", action_selector="multinomial"), 9, 12, "device"),
    "pi_logits_test": ("2s3z", dict(agent_output_type="pi_logits", action_selector="multinomial"), 7, 12, "device"),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(MAC_CASES))
def test_mac_unroll_gradients_match_float64(case):
    from cuda_utils import to_batch
    shape_key, over, B, T, layout = MAC_CASES[case]
    shape = SMAC_SHAPES[shape_key]
    N, A = shape.n_agents, shape.n_actions
    args = agent_args(shape, **over)
    la, aid, H = args.obs_last_action, args.obs_agent_id, args.rnn_hidden_dim
    pi, test_mode = args.agent_output_type == "pi_logits", case == "pi_logits_test"
    T_full = T + 5 if layout == "view" else T
    fields = numpy_episode_fields(shape, B, T_full, seed=11, ragged=True)
    scheme, groups = make_scheme(shape)
    mac = mac_REGISTRY["basic_mac"](scheme, groups, args)
    d_in = mac.agent.d_in
    load_agent(mac.agent, d_in, H, A, seed=5)
    mac.cuda()
    mac.action_selector.epsilon = 0.3
    batch = to_batch(shape, {k: v for k, v in fields.items() if k != "actions_onehot"},
                     device="cpu" if layout == "host" else "cuda")
    if layout == "view":
        batch = batch[:, :T]
        fields = {k: v[:, :T] for k, v in fields.items()}
    if layout == "compact":                 # bf16 obs, uint8 avail: converted for steps t-1 and t by the autograd path
        td = batch.data.transition_data
        td["obs"] = td["obs"].to(th.bfloat16)
        td["avail_actions"] = td["avail_actions"].to(th.uint8)
        fields = dict(fields, obs=td["obs"].float().cpu().numpy())
    w = np.random.default_rng(2).standard_normal((T, B, N, A))
    mac.init_hidden(B)
    loss = 0
    for t in range(T):
        out = mac.forward(batch, t, test_mode=test_mode)
        loss = loss + (out * th.tensor(w[t], dtype=th.float32, device=out.device)).sum()
    loss.backward()

    ref = ref_of(mac.agent, RefAgent(d_in, H, A))
    h = th.zeros(B * N, H, dtype=th.float64)
    loss_ref = 0
    for t in range(T):
        q, h = ref(ref_inputs(fields, t, N, A, la, aid), h)
        if pi:
            q = ref_policy(q, th.from_numpy(fields["avail_actions"][:, t]).reshape(B * N, A), 0.3, test_mode)
        loss_ref = loss_ref + (q.view(B, N, A) * th.from_numpy(w[t])).sum()
    loss_ref.backward()
    errs = grad_errs(mac.agent.named_parameters(), dict(ref.named_parameters()))
    print(case, {k: "%.1e" % v for k, v in errs.items()})
    assert all(e < 2e-5 for e in errs.values()), errs


@pytest.mark.gpu
@pytest.mark.parametrize("E", [32, 20])
def test_qmixer_gradients_match_float64(E):
    shape = SMAC_SHAPES["2s3z"]
    N, S = shape.n_agents, shape.state_dim
    args = default_args(shape, mixing_embed_dim=E, autograd_modules=True)
    th.manual_seed(E)
    mixer = QMixer(args).cuda()
    ref = ref_of(mixer, RefQMixer(S, N, E))
    rng = np.random.default_rng(E)
    qs, st, w = rng.standard_normal((6, 9, N)), rng.standard_normal((6, 9, S)), rng.standard_normal((6, 9, 1))
    qd = th.tensor(qs, dtype=th.float32, device="cuda", requires_grad=True)
    y = mixer(qd, th.tensor(st, dtype=th.float32, device="cuda"))
    (y * th.tensor(w, dtype=th.float32, device="cuda")).sum().backward()
    qr = th.tensor(qs, requires_grad=True)
    (ref(qr, th.tensor(st)) * th.tensor(w)).sum().backward()
    errs = {"q_tot": rel_err(y.detach().cpu(), ref(th.tensor(qs), th.tensor(st)).detach()), "agent_qs": rel_err(qd.grad.cpu(), qr.grad)}
    errs.update(grad_errs(mixer.named_parameters(), dict(ref.named_parameters())))
    print(E, {k: "%.1e" % v for k, v in errs.items()})
    assert all(e < 1e-5 for e in errs.values()), errs
    with pytest.raises(_lib.PmbError, match="states"):
        mixer(qd, th.zeros(6, 9, S, device="cuda", requires_grad=True))

    vq = th.tensor(qs, dtype=th.float32, device="cuda", requires_grad=True)
    (VDNMixer()(vq, None) * th.tensor(w, dtype=th.float32, device="cuda")).sum().backward()
    assert rel_err(vq.grad.cpu(), np.broadcast_to(w, qs.shape)) < 1e-7


# ---- GPU: a custom learner against the fused learner step --------------------------------------------------------------
def custom_q_learner_backward(mac, target_mac, mixer, target_mixer, batch, args):
    """learners/q_learner.py:37-103 up to loss.backward(), on this package's modules; returns (loss, mask sum, cur_max)."""
    rewards = batch["reward"][:, :-1]
    actions = batch["actions"][:, :-1]
    terminated = batch["terminated"][:, :-1].float()
    mask = batch["filled"][:, :-1].float()
    mask[:, 1:] = mask[:, 1:] * (1 - terminated[:, :-1])
    avail_actions = batch["avail_actions"]
    mac_out = []
    mac.init_hidden(batch.batch_size)
    for t in range(batch.max_seq_length):
        mac_out.append(mac.forward(batch, t=t))
    mac_out = th.stack(mac_out, dim=1)
    chosen_action_qvals = th.gather(mac_out[:, :-1], dim=3, index=actions).squeeze(3)
    with th.no_grad():
        target_mac_out = []
        target_mac.init_hidden(batch.batch_size)
        for t in range(batch.max_seq_length):
            target_mac_out.append(target_mac.forward(batch, t=t))
        target_mac_out = th.stack(target_mac_out[1:], dim=1)
        target_mac_out[avail_actions[:, 1:] == 0] = -9999999
    cur_max = None
    if args.double_q:
        mac_out_detach = mac_out.clone().detach()
        mac_out_detach[avail_actions == 0] = -9999999
        cur_max = mac_out_detach[:, 1:].max(dim=3, keepdim=True)[1]
        target_max_qvals = th.gather(target_mac_out, 3, cur_max).squeeze(3)
    else:
        target_max_qvals = target_mac_out.max(dim=3)[0]
    if mixer is not None:
        chosen_action_qvals = mixer(chosen_action_qvals, batch["state"][:, :-1])
        with th.no_grad():
            target_max_qvals = target_mixer(target_max_qvals, batch["state"][:, 1:])
    targets = rewards + args.gamma * (1 - terminated) * target_max_qvals
    td_error = chosen_action_qvals - targets.detach()
    mask = mask.expand_as(td_error)
    loss = ((td_error * mask) ** 2).sum() / mask.sum()
    loss.backward()
    return loss, mask.sum(), cur_max


def fused_gradient(learner, batch):
    """pmb_qlearner_train_step with skip_update = 1: the flat gradient of sum((td * mask)^2), and the online Q."""
    a = learner.args
    f = learner._ensure_flat()
    dev = f["p"].device
    names = ["obs", "actions", "avail_actions", "reward", "terminated", "filled"] + (["state"] if a.mixer == "qmix" else [])
    fields, _, B, T = learner._step_fields(batch, names, dev, False)
    S = fields["state"].shape[-1] if "state" in fields else 1
    dims = learner._layout_dims(B=B, T=T, O=fields["obs"].shape[3], S=S)
    keep = []
    pb = _lib.make_batch(fields, need_state=a.mixer == "qmix", keep=keep, dims=dims, entry=_lib.ENTRY_TRAIN_STEP)
    need = learner._ensure_workspace(dims, dev)
    hp = _lib.HParams(a.gamma, a.lr, a.optim_alpha, a.optim_eps, a.grad_norm_clip, 0, 1, 0)
    _lib.check(_lib.lib().pmb_qlearner_train_step(C.byref(dims), C.byref(pb), C.byref(hp), _lib.ptr(f["p"]), _lib.ptr(f["g"]),
                                                  _lib.ptr(f["sq"]), _lib.ptr(f["target"]), _lib.ptr(learner._workspace), need,
                                                  _lib.ptr(learner._stats), _lib.stream_ptr(dev)), "pmb_qlearner_train_step")
    q_on = learner.workspace_views(dims)["q_on"].view(T, B, a.n_agents, a.n_actions).permute(1, 0, 2, 3)
    return f["g"][:f["layout"].n_total].clone(), q_on.clone()


# id: (shape, mixer, double_q, B, T, seed).  With double_q the seeds are chosen so that every arg-max on an unmasked step
# has a top-2 gap above 1e-3 max|Q| in float64 (checked below at 1e-4 on the GPU's Q), as tests/test_config_matrix.py does
# for the rollout: a near-tie would pick a different target in the two fp32 paths.
LEARNER_CASES = {
    "3m_qmix_double": ("3m", "qmix", True, 12, 20, 9),
    "3m_vdn": ("3m", "vdn", False, 12, 20, 4),
    "2s3z_qmix": ("2s3z", "qmix", False, 8, 16, 5),
    "2s3z_vdn_double": ("2s3z", "vdn", True, 8, 16, 8),
    "2s3z_qmix_b32": ("2s3z", "qmix", False, 32, 16, 7),            # 160 rows: sliced weight gradients
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(LEARNER_CASES))
def test_custom_learner_equals_fused_step(case):
    from cuda_utils import build_learner, to_batch
    shape_key, mixer_name, double_q, B, T, seed = LEARNER_CASES[case]
    shape = SMAC_SHAPES[shape_key]
    args = default_args(shape, mixer=mixer_name, double_q=double_q, learner_log_interval=0, grad_norm_clip=1e30)
    rng = np.random.default_rng(seed)
    d_in = shape.obs_dim + shape.n_actions + shape.n_agents
    agent = orc.init_params(orc.agent_param_shapes(d_in, 64, shape.n_actions), rng)
    target = {k: (v + 0.05 * rng.standard_normal(v.shape)).astype(np.float32) for k, v in agent.items()}
    mix = orc.init_params(orc.qmix_param_shapes(shape.state_dim, shape.n_agents, 32), rng) if mixer_name == "qmix" else None
    tmix = {k: (v + 0.02 * rng.standard_normal(v.shape)).astype(np.float32) for k, v in mix.items()} if mix else None
    fields = numpy_episode_fields(shape, B, T, seed=seed + 100, ragged=True)
    batch = to_batch(shape, fields)
    learner, _ = build_learner(shape, copy.copy(args), agent, target, mix, tmix)
    g_fused, q_on = fused_gradient(learner, batch)

    # the custom learner: its own modules with the key on, loaded with the same parameters
    ca = copy.copy(args)
    ca.autograd_modules = True
    ca.device = "cuda"
    scheme, groups = make_scheme(shape)
    mac = mac_REGISTRY["basic_mac"](scheme, groups, ca)
    mac.agent.load_state_dict(learner.mac.agent.state_dict())
    mac.cuda()
    target_mac = copy.deepcopy(mac)
    target_mac.agent.load_state_dict(learner.target_mac.agent.state_dict())
    mixer = target_mixer = None
    if mixer_name == "qmix":
        mixer = QMixer(ca).cuda()
        mixer.load_state_dict(learner.mixer.state_dict())
        target_mixer = QMixer(ca).cuda()
        target_mixer.load_state_dict(learner.target_mixer.state_dict())
    elif mixer_name == "vdn":
        mixer = target_mixer = VDNMixer()
    loss, mask_sum, cur_max = custom_q_learner_backward(mac, target_mac, mixer, target_mixer, batch, ca)

    if double_q:
        live = batch["filled"][:, :-1, 0].float()
        live[:, 1:] *= 1 - batch["terminated"][:, :-2, 0].float()
        live = live.bool()                                   # the steps the loss masks in
        qf = q_on.masked_fill(batch["avail_actions"] == 0, -9999999.0)[:, 1:]
        top2 = qf.topk(2, dim=3)[0]
        gap = (top2[..., 0] - top2[..., 1])[live]
        assert gap.min().item() > 1e-4 * q_on.abs().max().item(), gap.min().item()
        assert th.equal(qf.argmax(3)[live], cur_max[..., 0][live])

    named = [("agent." + k, p) for k, p in mac.agent.named_parameters()]
    if mixer_name == "qmix":
        named += [("mixer." + k, p) for k, p in mixer.named_parameters()]
    fused_named = dict([("agent." + k, p) for k, p in learner.mac.agent.named_parameters()] +
                       ([("mixer." + k, p) for k, p in learner.mixer.named_parameters()] if mixer_name == "qmix" else []))
    base = learner._flat["p"].data_ptr()
    errs = {}
    for k, p in named:
        fp = fused_named[k]
        off = (fp.data_ptr() - base) // 4
        g_ref = g_fused[off:off + fp.numel()].view(fp.shape)
        errs[k] = rel_err((p.grad * mask_sum).detach().cpu().numpy(), g_ref.cpu().numpy())
    print(case, "loss %.4f" % loss.item(), {k: "%.1e" % v for k, v in errs.items()})
    assert all(e < 2e-5 for e in errs.values()), errs


# ---- GPU: accumulation, optimiser steps, determinism, launch budget, double backward ----------------------------------
def _mac_and_batch(shape_key="3m", B=9, T=12, **over):
    from cuda_utils import to_batch
    shape = SMAC_SHAPES[shape_key]
    args = agent_args(shape, **over)
    scheme, groups = make_scheme(shape)
    mac = mac_REGISTRY["basic_mac"](scheme, groups, args)
    load_agent(mac.agent, mac.agent.d_in, args.rnn_hidden_dim, shape.n_actions, seed=9)
    mac.cuda()
    fields = numpy_episode_fields(shape, B, T, seed=12, ragged=True)
    return mac, to_batch(shape, {k: v for k, v in fields.items() if k != "actions_onehot"}), T


def _unroll_loss(mac, batch, T):
    mac.init_hidden(batch.batch_size)
    w = th.linspace(-1, 1, mac.args.n_actions, device="cuda")
    return sum((mac.forward(batch, t) * w).sum() * (1 + 0.1 * t) for t in range(T))


@pytest.mark.gpu
def test_gradients_accumulate_into_bound_views_and_after_set_to_none():
    """QLearner points .grad at views of its flat gradient buffer (flat.bind): AccumulateGrad adds into them in place;
    with the grads set to None it creates fresh ones; a torch optimiser step is seen by the next forward."""
    from cuda_utils import build_learner
    mac, batch, T = _mac_and_batch()
    params = list(mac.agent.parameters())
    _unroll_loss(mac, batch, T).backward()
    g1 = [p.grad.clone() for p in params]

    learner, _ = build_learner(SMAC_SHAPES["3m"], default_args(SMAC_SHAPES["3m"], autograd_modules=True))
    lmac = learner.mac
    lmac.agent.load_state_dict(mac.agent.state_dict())
    flat_g = learner._flat["g"]
    flat_g.fill_(0.5)
    for p in lmac.agent.parameters():
        assert p.grad is not None and p.grad.data_ptr() >= flat_g.data_ptr()
    _unroll_loss(lmac, batch, T).backward()
    for p, g in zip(lmac.agent.parameters(), g1):
        assert rel_err(p.grad.cpu(), (g + 0.5).cpu()) < 1e-6
        assert flat_g.data_ptr() <= p.grad.data_ptr() < flat_g.data_ptr() + 4 * flat_g.numel()

    for p in params:
        p.grad = None                                       # zero_grad(set_to_none=True)
    _unroll_loss(mac, batch, T).backward()
    _unroll_loss(mac, batch, T).backward()
    for p, g in zip(params, g1):
        assert rel_err(p.grad.cpu(), (2 * g).cpu()) < 1e-6

    opt = th.optim.SGD(params, lr=0.05)
    opt.step()
    opt.zero_grad(set_to_none=True)
    mac.init_hidden(batch.batch_size)
    with th.no_grad():
        q_after = mac.forward(batch, 0).clone()
    ref = ref_of(mac.agent, RefAgent(mac.agent.d_in, 64, mac.args.n_actions))
    x0 = batch["obs"][:, 0].cpu().double()
    B, N = x0.shape[:2]
    x0 = th.cat([x0, th.zeros(B, N, mac.args.n_actions, dtype=th.float64), th.eye(N, dtype=th.float64).expand(B, N, N)], -1)
    q_ref, _ = ref(x0.reshape(B * N, -1), th.zeros(B * N, 64, dtype=th.float64))
    assert rel_err(q_after.cpu().reshape(B * N, -1), q_ref.detach()) < 1e-5


@pytest.mark.gpu
def test_backward_is_deterministic_and_within_the_launch_budget():
    mac, batch, T = _mac_and_batch("2s3z", B=40, T=10)
    L = _lib.lib()
    params = list(mac.agent.parameters())
    th.cuda.synchronize()
    n0 = L.pmb_launch_count()
    loss = _unroll_loss(mac, batch, T)
    n1 = L.pmb_launch_count()
    g_a = th.autograd.grad(loss, params, retain_graph=True)
    n2 = L.pmb_launch_count()
    g_b = th.autograd.grad(loss, params)
    g_c = th.autograd.grad(_unroll_loss(mac, batch, T), params)
    print("launches per step: forward %.2f backward %.2f" % ((n1 - n0) / T, (n2 - n1) / T))
    assert (n1 - n0) <= 3 * T and (n2 - n1) <= 5 * T, (n1 - n0, n2 - n1)
    for a, b, c in zip(g_a, g_b, g_c):
        assert th.equal(a, b) and th.equal(a, c)


@pytest.mark.gpu
def test_double_backward_raises_a_clear_error():
    mac, batch, T = _mac_and_batch(T=3)
    with pytest.raises(_lib.PmbError, match="double backward"):
        _unroll_loss(mac, batch, T).backward(create_graph=True)
    args = default_args(SMAC_SHAPES["3m"], autograd_modules=True)
    mixer = QMixer(args).cuda()
    qs = th.randn(2, 3, 3, device="cuda", requires_grad=True)
    with pytest.raises(_lib.PmbError, match="double backward"):
        mixer(qs, th.randn(2, 3, 48, device="cuda")).sum().backward(create_graph=True)
