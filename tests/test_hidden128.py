"""rnn_hidden_dim = 128 on both precision tiers against the float64 oracle.

At H = 128 the agent's GRU runs split (csrc/gru_h128.cu): the input gates of all timesteps as one GEMM, a recurrence
kernel with only W_hh on chip, fc2 as one GEMM; in the backward a BPTT kernel with only W_hh on chip and the fc1-output
gradient as one GEMM plus the ReLU mask.  Checked here through every entry point that takes rnn_hidden_dim:
1. the learner step, with the protocol and bounds of test_config_matrix.test_learner_step_matches_oracle (clip off,
   RMSprop pre-warmed to 1e-2, target nets perturbed, ragged batches; fp32: Q 1e-5, stats 2e-5, gradients 2e-5,
   parameters 5e-5; bf16: gradients and updates 1e-2 relative L2 with the decisions the step takes on bf16 operands
   pinned: the double-Q arg-max and, where the tensor-core mixer runs, the hypernet signs), and two consecutive fp32
   steps with a target sync between them;
2. three BasicMAC rollout steps with injected epsilon-draws, 19 envs of 27 agents (513 rows: not a multiple of the
   recurrence kernel's 64-row tile);
3. one COMA train step on the fp32 tier at the bounds of test_coma_gpu;
4. host only: the workspace sizes, the refusal of other widths, the formats only the H = 64 tensor-core path reads.
"""
import copy
import ctypes as C

import numpy as np
import pytest
import torch as th

from golden_utils import rel_err
from oracle import coma_oracle as co, qlearner_oracle as orc
from pymarl_b200 import _lib
from pymarl_b200.synthetic import SMAC_SHAPES, default_args, numpy_episode_fields
from test_config_matrix import STATS, TOL_BF16, _l2, _oracle_learner

H = 128
# id: (shape, mixer, overrides, B, T)
LEARNER_CASES = {
    "qmix_3m": ("3m", "qmix", {}, 32, 20),
    "vdn_MMM2_no_agent_id": ("MMM2", "vdn", dict(obs_agent_id=False), 16, 14),
    "iql_2s3z_no_double_q": ("2s3z", None, dict(double_q=False), 24, 16),
}
FP32_BOUNDS = {"q": 1e-5, "stat": 2e-5, "grad": 2e-5, "param": 5e-5}
BF16_BOUNDS = {"q": TOL_BF16, "stat": TOL_BF16, "grad": TOL_BF16, "upd": TOL_BF16}


def _args(case, precision, **more):
    shape, mixer, over, _, _ = LEARNER_CASES[case]
    return default_args(SMAC_SHAPES[shape], mixer=mixer, learner_log_interval=0, precision=precision, grad_norm_clip=1e30,
                        rnn_hidden_dim=H, **over, **more)


def _dims(shape, args, B=8, T=4, precision="fp32", H_=H):
    return _lib.make_dims(B, T, shape.n_agents, shape.obs_dim, shape.state_dim, shape.n_actions, H_, args.mixing_embed_dim,
                          obs_last_action=args.obs_last_action, obs_agent_id=args.obs_agent_id, mixer=args.mixer,
                          double_q=args.double_q, precision=precision)


def _gpu_params(learner):
    named = {("agent." + k): v for k, v in learner.mac.agent.named_parameters()}
    if learner.mixer is not None:
        named.update({("mixer." + k): v for k, v in learner.mixer.named_parameters()})
    return named


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("case", list(LEARNER_CASES))
def test_learner_step_matches_oracle(case, precision):
    from cuda_utils import build_learner, gpu_decisions, to_batch
    shape_key, mixer, _, B, T = LEARNER_CASES[case]
    shape = SMAC_SHAPES[shape_key]
    args = _args(case, precision)
    fields = numpy_episode_fields(shape, B, T, seed=41, ragged=True)
    base = _oracle_learner(shape, copy.copy(args), seed=17, dtype=np.float32)
    dec = None
    if precision == "bf16":
        tc_mixer = _lib.field_dtype_supported(_dims(shape, args, B, T, "bf16"), _lib.ENTRY_TRAIN_STEP, "state",
                                              _lib.DTYPE_BF16)
        which = (("hypernet",) if tc_mixer else ()) + (("cur_max",) if args.double_q else ())
        dec = gpu_decisions(shape, args, base, fields, which=which) if which else None

    o = _oracle_learner(shape, copy.copy(args), seed=17, dtype=np.float64)
    p0 = {("agent." + k): v.copy() for k, v in o.agent.items()}
    p0.update({("mixer." + k): v.copy() for k, v in o.mixer_p.items()})
    f64 = {k: (v.astype(np.float64) if v.dtype == np.float32 else v) for k, v in fields.items()}
    stats, g_ref, fw = o.train(f64, 0, 0, decisions=dec)
    p1 = {("agent." + k): v for k, v in o.agent.items()}
    p1.update({("mixer." + k): v for k, v in o.mixer_p.items()})

    a = copy.copy(args)
    a.keep_q = 1
    learner, _ = build_learner(shape, a, base.agent, base.target_agent, base.mixer_p, base.target_mixer_p)
    learner._flat["sq"].fill_(1e-2)
    flat0 = learner._flat["p"].clone()
    learner.train(to_batch(shape, fields), 0, 0)
    assert learner._last_dims.H == H
    st = learner.stats()
    ws = learner.workspace_views(learner._last_dims)
    q = ws["q_on"].view(T, B, shape.n_agents, -1).permute(1, 0, 2, 3).cpu().numpy()
    named = _gpu_params(learner)
    assert sorted(named) == sorted(g_ref)
    base_ptr = learner._flat["p"].data_ptr()
    report = {"q": rel_err(q, fw["mac_out"])}
    report.update({"stat." + k: abs(st[k] - stats[k]) / max(1.0, abs(stats[k])) for k in STATS})
    for k, prm in named.items():
        off = (prm.data_ptr() - base_ptr) // 4
        g_gpu = prm.grad.cpu().numpy().astype(np.float64)
        p_gpu = prm.detach().cpu().numpy().astype(np.float64)
        u_gpu = p_gpu - flat0[off:off + prm.numel()].view(prm.shape).double().cpu().numpy()
        assert np.abs(p1[k] - p0[k]).max() > 0, k
        if precision == "fp32":
            report["grad." + k] = rel_err(g_gpu, g_ref[k])
            report["param." + k] = rel_err(p_gpu, p1[k])
        else:
            report["grad." + k] = _l2(g_gpu, g_ref[k])
            report["upd." + k] = _l2(u_gpu, p1[k] - p0[k])
    print(case, precision, {k: "%.1e" % v for k, v in report.items()})
    bounds = FP32_BOUNDS if precision == "fp32" else BF16_BOUNDS
    for k, e in report.items():
        assert e < bounds[k.split(".")[0]], (case, precision, k, e)


@pytest.mark.gpu
def test_two_steps_across_a_target_sync_match_oracle():
    """QMIX on 3m, fp32 tier: the first step ends with a target sync (target_update_interval = 1, episode 1), so the second
    step's target pass runs on the nets the first step wrote.  Stats of both steps and the parameters after each."""
    from cuda_utils import build_learner, to_batch
    case = "qmix_3m"
    shape_key, _, _, B, T = LEARNER_CASES[case]
    shape = SMAC_SHAPES[shape_key]
    args = _args(case, "fp32", target_update_interval=1)
    fields = [numpy_episode_fields(shape, B, T, seed=s, ragged=True) for s in (41, 42)]
    base = _oracle_learner(shape, copy.copy(args), seed=17, dtype=np.float32)
    o = _oracle_learner(shape, copy.copy(args), seed=17, dtype=np.float64)
    learner, _ = build_learner(shape, copy.copy(args), base.agent, base.target_agent, base.mixer_p, base.target_mixer_p)
    learner._flat["sq"].fill_(1e-2)
    for step, f in enumerate(fields):
        stats, _, _ = o.train({k: (v.astype(np.float64) if v.dtype == np.float32 else v) for k, v in f.items()}, step, 1)
        learner.train(to_batch(shape, f), step, 1)
        st = learner.stats()
        report = {"stat." + k: abs(st[k] - stats[k]) / max(1.0, abs(stats[k])) for k in STATS}
        ref = {("agent." + k): v for k, v in o.agent.items()}
        ref.update({("mixer." + k): v for k, v in o.mixer_p.items()})
        for k, prm in _gpu_params(learner).items():
            report["param." + k] = rel_err(prm.detach().cpu().numpy(), ref[k])
        print(step, {k: "%.1e" % v for k, v in report.items()})
        for k, e in report.items():
            assert e < FP32_BOUNDS[k.split(".")[0]], (step, k, e)
    assert o.n_target_updates == 1 and learner.last_target_update_episode == 1


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_rollout_steps_match_oracle(precision):
    """As test_config_matrix.test_rollout_steps_match_oracle: Q and hidden state within the tier's tolerance, the random
    actions equal, the greedy ones wherever the oracle's best-to-second gap exceeds twice the tolerance times max|Q|."""
    from cuda_utils import to_batch
    from pymarl_b200 import mac_REGISTRY
    from pymarl_b200.synthetic import make_scheme
    shape, envs = SMAC_SHAPES["27m_vs_30m"], 19
    N, A = shape.n_agents, shape.n_actions
    args = default_args(shape, device="cuda", precision=precision, rnn_hidden_dim=H)
    scheme, groups = make_scheme(shape)
    mac = mac_REGISTRY["basic_mac"](scheme, groups, args)
    mac.cuda()
    rng = np.random.default_rng(6)
    agent = orc.init_params(orc.agent_param_shapes(shape.obs_dim + A + N, H, A), rng)
    mac.agent.load_state_dict({k: th.from_numpy(v) for k, v in agent.items()})
    p64 = {k: v.astype(np.float64) for k, v in agent.items()}
    fields = numpy_episode_fields(shape, envs, 5, seed=4, ragged=False)
    batch = to_batch(shape, {k: v for k, v in fields.items() if k != "actions_onehot"})
    sel = mac.action_selector
    seen = []
    select = sel.select_action
    sel.select_action = lambda q, *a, **kw: (seen.append(q.detach().clone()), select(q, *a, **kw))[1]
    mac.init_hidden(envs)
    h = np.zeros((envs * N, H))
    tol = 1e-5 if precision == "fp32" else TOL_BF16
    for t in range(3):
        u = rng.random((envs, N), dtype=np.float32)
        expo = rng.exponential(size=(envs * N, A)).astype(np.float32)
        sel.draw = lambda q, u=th.from_numpy(u).cuda(), e=th.from_numpy(expo).cuda(): (u, e)
        acts = mac.select_actions(batch, t_ep=t, t_env=40000).cpu().numpy()
        eps = sel.epsilon
        a_ref, q_ref, h = orc.mac_select_actions(p64, fields, t, h, eps, u, expo.reshape(envs, N, A), True, True)
        q = seen[-1].cpu().numpy().reshape(q_ref.shape)
        hid = mac.hidden_states.detach().cpu().numpy().reshape(h.shape)
        print(precision, t, "q %.1e hidden %.1e" % (rel_err(q, q_ref), rel_err(hid, h)))
        assert rel_err(q, q_ref) < tol, (t, rel_err(q, q_ref))
        assert rel_err(hid, h) < tol, (t, rel_err(hid, h))
        random = u < np.float32(eps)
        avail = fields["avail_actions"][:, t]
        top2 = np.sort(np.where(avail == 0, -np.inf, q_ref), axis=2)[..., -2:]
        clear = top2[..., 1] - top2[..., 0] > 2 * tol * np.abs(q_ref).max()
        assert random.any() and (~random & clear).mean() > 0.5 * (~random).mean(), t
        np.testing.assert_array_equal(acts[random], a_ref[random])
        np.testing.assert_array_equal(acts[~random & clear], a_ref[~random & clear])


@pytest.mark.gpu
def test_rnn_agent_forward_matches_oracle():
    """RNNAgent.forward (pmb_agent_fc1_dense_fwd + pmb_agent_gru_unroll_fwd with a gates buffer) on a dense input."""
    from types import SimpleNamespace
    from pymarl_b200.modules.agents.rnn_agent import RNNAgent
    rows, d_in, A = 77, 40, 9
    rng = np.random.default_rng(3)
    p = orc.init_params(orc.agent_param_shapes(d_in, H, A), rng)
    agent = RNNAgent(d_in, SimpleNamespace(rnn_hidden_dim=H, n_actions=A)).cuda()
    agent.load_state_dict({k: th.from_numpy(v) for k, v in p.items()})
    x = rng.standard_normal((rows, d_in)).astype(np.float32)
    h0 = (0.5 * rng.standard_normal((rows, H))).astype(np.float32)
    q, h = agent(th.from_numpy(x).cuda(), th.from_numpy(h0).cuda())
    f = {k: v.astype(np.float64) for k, v in p.items()}
    xr = np.maximum(x @ f["fc1.weight"].T + f["fc1.bias"], 0)
    gi, gh = xr @ f["rnn.weight_ih"].T + f["rnn.bias_ih"], h0 @ f["rnn.weight_hh"].T + f["rnn.bias_hh"]
    sig = lambda v: 1 / (1 + np.exp(-v))
    r, z = sig(gi[:, :H] + gh[:, :H]), sig(gi[:, H:2 * H] + gh[:, H:2 * H])
    n = np.tanh(gi[:, 2 * H:] + r * gh[:, 2 * H:])
    h_ref = (1 - z) * n + z * h0
    assert rel_err(h.cpu().numpy(), h_ref) < 1e-5
    assert rel_err(q.cpu().numpy(), h_ref @ f["fc2.weight"].T + f["fc2.bias"]) < 1e-5


@pytest.mark.gpu
def test_coma_train_step_matches_oracle():
    """test_coma_gpu.test_coma_train_step_matches_oracle's 2s3z-8-12 case at H = 128: one COMALearner.train on a ragged
    batch against the float64 oracle at TRAIN_BOUNDS."""
    from cuda_utils import to_batch
    from test_coma_gpu import COMA_KW, TRAIN_BOUNDS, build_coma, state_np
    shape, B, T = SMAC_SHAPES["2s3z"], 8, 12
    N, A = shape.n_agents, shape.n_actions
    args = default_args(shape, mixer=None, rnn_hidden_dim=H, **COMA_KW)
    rng = np.random.default_rng(5)
    agent = orc.init_params(orc.agent_param_shapes(shape.obs_dim + A + N, H, A), rng)
    crit = co.init_critic(co.critic_param_shapes(shape.state_dim, shape.obs_dim, N, A), rng)
    tcrit = {k: (v + 0.05 * rng.standard_normal(v.shape)).astype(np.float32) for k, v in crit.items()}
    fields = numpy_episode_fields(shape, B, T, seed=17, ragged=True)
    for k in fields:
        fields[k][:, T - 3:] = 0
    f64 = lambda p: {k: v.astype(np.float64) for k, v in p.items()}
    olr = co.OracleCOMALearner(f64(agent), f64(crit), copy.copy(args))
    olr.target_critic = f64(tcrit)
    learner, logger = build_coma(shape, args, agent, crit, tcrit)
    eps = 0.37
    learner.mac.action_selector.epsilon = eps
    st, _, fw = olr.train(fields, 0, 0, float(np.float32(eps)))
    learner.train(to_batch(shape, fields), 0, 0)
    ws = learner.workspace_views()
    err = {"targets": rel_err(ws["targets"].cpu().numpy(), fw["targets"]),
           "pi": rel_err(ws["pi"].view(T - 1, B, N, A).permute(1, 0, 2, 3).cpu().numpy(), fw["pi"])}
    rel = lambda got, ref: float(np.max(np.abs(np.asarray(got) - ref) / np.maximum(1.0, np.abs(ref))))
    for k in ("critic_loss", "critic_grad_norm", "td_error_abs", "q_taken_mean", "target_mean"):
        err["stat." + k] = rel(logger.stats[k][-1][1], st[k])
    for k in ("advantage_mean", "coma_loss", "agent_grad_norm", "pi_max"):
        err["agent_stat." + k] = rel(logger.stats[k][-1][1], st[k])
    for tag, mod, ref in (("agent", learner.mac.agent, olr.agent), ("critic", learner.critic, olr.critic)):
        got = state_np(mod)
        for k, v in ref.items():
            err["param.%s.%s" % (tag, k)] = rel_err(got[k], v)
    print({k: "%.1e" % v for k, v in err.items()})
    for k, e in err.items():
        group = k.split(".")[0] if not k.startswith("param.") else ".".join(k.split(".")[:2])
        assert e < TRAIN_BOUNDS[group], (k, e)


def test_workspace_sizes_and_refusals():
    """Host only (no device call)."""
    L = _lib.lib()
    shape = SMAC_SHAPES["27m_vs_30m"]
    for precision in ("fp32", "bf16"):
        args = default_args(shape, mixer="qmix", precision=precision, rnn_hidden_dim=H)
        d, d64 = _dims(shape, args, 1024, 180, precision), _dims(shape, args, 1024, 180, precision, H_=64)
        learner = L.pmb_learner_workspace_bytes(C.byref(d))
        # the fp32 activations: x_on, x_tg, h_stash and gates are [T][R][H], [T][R][H], [T+1][R][H], [T][R][4H]
        assert learner >= 4 * 180 * 1024 * 27 * 7 * H > 0
        assert learner > L.pmb_learner_workspace_bytes(C.byref(d64)) > 0
        # the rollout step adds the input-gate buffer [R][3H]
        assert L.pmb_select_actions_workspace_bytes(C.byref(d)) >= 4 * 1024 * 27 * 4 * H
        coma = _dims(shape, default_args(shape, mixer=None, precision=precision), 8, 120, precision)
        coma.E = 128
        assert L.pmb_coma_workspace_bytes(C.byref(coma)) > 0
        # formats read only by the H = 64 tensor-core path
        for entry in (_lib.ENTRY_TRAIN_STEP, _lib.ENTRY_SELECT_ACTIONS):
            assert not _lib.obs_bf16_supported(d, entry)
            assert not _lib.field_dtype_supported(d, entry, "avail_actions", _lib.DTYPE_U8)
    bad = _dims(shape, default_args(shape, mixer="qmix"), H_=96)
    assert L.pmb_learner_workspace_bytes(C.byref(bad)) == -1
    with pytest.raises(_lib.PmbError, match=r"rnn_hidden_dim 96 unsupported \(16, 32, 64, 128\)"):
        _lib.flat_layout(bad)
