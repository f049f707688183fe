"""The reference's configuration keys off their defaults - double_q, obs_last_action, obs_agent_id, rnn_hidden_dim,
mixing_embed_dim - and n_actions above 64, on both precision tiers, against the float64 oracle.

A user sets these keys in YAML and QLearner passes them to the kernels unchecked.  Each case below is the only test of one
branch of the tier it runs on (the last column of LEARNER_CASES):
1. the learner step, one case per branch: clip off so the gradients compare directly, RMSprop state pre-warmed to 1e-2 on
   both sides, target nets perturbed, ragged batches.
   fp32 tier: Q 1e-5, stats 2e-5, every gradient 2e-5 (max-norm relative), post-update parameters 5e-5.
   bf16 tier: every gradient and every update within 1e-2 (relative L2) of the float64 oracle run with the GPU's decisions
   pinned, stats within 1e-2.  Only the decisions the step takes on bf16 operands are pinned: the fc1 ReLU mask where the
   tensor-core agent runs, the hypernet signs and the V ReLU where the tensor-core mixer runs, the double-Q arg-max
   whenever double_q is on.  Elsewhere the forward is fp32 and the oracle keeps its own decisions.
2. three consecutive BasicMAC rollout steps with injected epsilon-draws against the oracle MAC.
3. a host-only guard: every case takes the dispatch path it claims (tensor-core agent, tensor-core mixer, fused streaming
   learner step, tensor-core rollout), so a moved dispatch condition fails here instead of quietly testing another path.
"""
import copy

import numpy as np
import pytest
import torch as th

from golden_utils import rel_err
from oracle import qlearner_oracle as orc
from pymarl_b200 import _lib
from pymarl_b200.synthetic import SMAC_SHAPES, SmacShape, default_args, numpy_episode_fields

NO_FOLD = SmacShape("no_fold", 10, 120, 64, 9, 21)    # 64 * ceil(O / 64) - O < N + 1: agent-id table in the fc1 epilogue
WIDE_A = SmacShape("wide_a", 4, 40, 52, 70, 6)        # A > 64: the agent runs off the tensor-core kernels
TOL_BF16 = 1e-2

# id: (shape, mixer, overrides, B, T, bf16 path it pins)
LEARNER_CASES = {
    "no_double_q": ("2s3z", "qmix", dict(double_q=False), 24, 16, "fused q-select with double_q = 0"),
    "no_last_action": ("3m", "qmix", dict(obs_last_action=False), 32, 20, "fused; pack, tables and dW without the act block"),
    "no_agent_id": ("MMM2", "vdn", dict(obs_agent_id=False), 16, 14, "fused; folded id columns zero, bias column kept"),
    "no_inputs_no_double": ("27m_vs_30m", None, dict(obs_last_action=False, obs_agent_id=False, double_q=False), 8, 12,
                            "fused IQL"),
    "nofold_no_last_action": (NO_FOLD, "qmix", dict(obs_last_action=False), 21, 16,
                              "id table in the fc1 epilogue, scatter grads"),
    "h32": ("3m", "qmix", dict(rnn_hidden_dim=32), 32, 20, "CUDA-core agent + tc mixer"),
    "h16_vdn": ("2s3z", "vdn", dict(rnn_hidden_dim=16), 24, 16, "CUDA-core agent"),
    "e64": ("3m", "qmix", dict(mixing_embed_dim=64), 32, 20, "tc agent + CUDA-core mixer, E > 32"),
    "e20": ("2s3z", "qmix", dict(mixing_embed_dim=20), 24, 16, "tc agent + CUDA-core mixer, E not a multiple of 8"),
    "a70": (WIDE_A, "qmix", {}, 24, 12, "CUDA-core agent (A > 64) + tc mixer"),
}

# id: (shape, overrides, envs)
ROLLOUT_CASES = {
    "no_last_action": ("3m", dict(obs_last_action=False), 37),
    "no_agent_id": ("MMM2", dict(obs_agent_id=False), 23),
    "no_inputs": ("27m_vs_30m", dict(obs_last_action=False, obs_agent_id=False), 19),
    "h32": ("3m", dict(rnn_hidden_dim=32), 37),
    "a70": (WIDE_A, {}, 29),
}

# the bf16-tier path of every case: (tensor-core agent, tensor-core mixer, fused streaming learner step, tensor-core rollout)
PATHS = {
    "no_double_q": (True, True, True, True),
    "no_last_action": (True, True, True, True),
    "no_agent_id": (True, False, True, True),
    "no_inputs_no_double": (True, False, True, True),
    "nofold_no_last_action": (True, True, False, True),
    "h32": (False, True, False, False),
    "h16_vdn": (False, False, False, False),
    "e64": (True, False, False, True),
    "e20": (True, False, False, True),
    "a70": (False, True, False, False),
    "rollout/no_last_action": (True, True, True, True),
    "rollout/no_agent_id": (True, True, True, True),
    "rollout/no_inputs": (True, True, True, True),
    "rollout/h32": (False, True, False, False),
    "rollout/a70": (False, True, False, False),
}


def _shape(s):
    return SMAC_SHAPES[s] if isinstance(s, str) else s


def _learner_args(case, precision):
    shape, mixer, over, _, _, _ = LEARNER_CASES[case]
    return default_args(_shape(shape), mixer=mixer, learner_log_interval=0, precision=precision, grad_norm_clip=1e30,
                        **over)


def _bf16_paths(shape, args, B=64, T=20):
    d = _lib.make_dims(B, T, shape.n_agents, shape.obs_dim, shape.state_dim, shape.n_actions, args.rnn_hidden_dim,
                       args.mixing_embed_dim, obs_last_action=args.obs_last_action, obs_agent_id=args.obs_agent_id,
                       mixer=args.mixer, double_q=args.double_q, precision="bf16")
    sup = _lib.field_dtype_supported
    return (sup(d, _lib.ENTRY_TRAIN_STEP, "avail_actions", _lib.DTYPE_U8),
            sup(d, _lib.ENTRY_TRAIN_STEP, "state", _lib.DTYPE_BF16),
            _lib.obs_bf16_supported(d, _lib.ENTRY_TRAIN_STEP),
            sup(d, _lib.ENTRY_SELECT_ACTIONS, "avail_actions", _lib.DTYPE_U8))


def test_each_case_takes_the_path_it_claims():
    """Host only (no device call): the dispatch predicates of pmb_field_dtype_supported / pmb_obs_bf16_supported."""
    got = {}
    for case, (shape, _, _, B, T, _) in LEARNER_CASES.items():
        got[case] = _bf16_paths(_shape(shape), _learner_args(case, "bf16"), B, T)
    for case, (shape, over, envs) in ROLLOUT_CASES.items():
        got["rollout/" + case] = _bf16_paths(_shape(shape), default_args(_shape(shape), precision="bf16", **over), envs, 4)
    assert got == PATHS


def _oracle_learner(shape, args, seed, dtype):
    """Oracle learner with perturbed target nets and RMSprop state pre-warmed to 1e-2; float32 values, held in `dtype`."""
    rng = np.random.default_rng(seed)
    d_in = shape.obs_dim + (shape.n_actions if args.obs_last_action else 0) + (shape.n_agents if args.obs_agent_id else 0)
    agent = orc.init_params(orc.agent_param_shapes(d_in, args.rnn_hidden_dim, shape.n_actions), rng)
    mixer = orc.init_params(orc.qmix_param_shapes(shape.state_dim, shape.n_agents, args.mixing_embed_dim), rng) \
        if args.mixer == "qmix" else {}
    lr = orc.OracleQLearner(agent, mixer, args)
    for k in lr.target_agent:
        lr.target_agent[k] = (lr.target_agent[k] + 0.05 * rng.standard_normal(lr.target_agent[k].shape)).astype(np.float32)
    for k in lr.target_mixer_p:
        lr.target_mixer_p[k] = (lr.target_mixer_p[k] + 0.02 * rng.standard_normal(lr.target_mixer_p[k].shape)).astype(np.float32)
    for d in (lr.agent, lr.mixer_p, lr.target_agent, lr.target_mixer_p, lr.sq_agent, lr.sq_mixer):
        for k in d:
            d[k] = d[k].astype(dtype)
    for sq in list(lr.sq_agent.values()) + list(lr.sq_mixer.values()):
        sq[...] = 1e-2
    return lr


def _l2(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))


STATS = ("loss", "grad_norm", "td_error_abs", "q_taken_mean", "target_mean")


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("case", list(LEARNER_CASES))
def test_learner_step_matches_oracle(case, precision):
    from cuda_utils import build_learner, gpu_decisions, to_batch
    shape_key, mixer, _, B, T, _ = LEARNER_CASES[case]
    shape = _shape(shape_key)
    args = _learner_args(case, precision)
    fields = numpy_episode_fields(shape, B, T, seed=41, ragged=True)
    base = _oracle_learner(shape, copy.copy(args), seed=17, dtype=np.float32)

    dec = None
    if precision == "bf16":
        tc_agent, tc_mixer = PATHS[case][:2]
        which = (("relu_mask",) if tc_agent else ()) + (("hypernet",) if tc_mixer else ()) + \
            (("cur_max",) if args.double_q else ())
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
    st = learner.stats()
    ws = learner.workspace_views(learner._last_dims)
    q = ws["q_on"].view(T, B, shape.n_agents, -1).permute(1, 0, 2, 3).cpu().numpy()
    named = {("agent." + k): v for k, v in learner.mac.agent.named_parameters()}
    if learner.mixer is not None:
        named.update({("mixer." + k): v for k, v in learner.mixer.named_parameters()})
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
    if precision == "fp32":
        bounds = {"q": 1e-5, "stat": 2e-5, "grad": 2e-5, "param": 5e-5}
    else:
        bounds = {"q": TOL_BF16, "stat": TOL_BF16, "grad": TOL_BF16, "upd": TOL_BF16}
    for k, e in report.items():
        assert e < bounds[k.split(".")[0]], (case, precision, k, e)


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("case", list(ROLLOUT_CASES))
def test_rollout_steps_match_oracle(case, precision):
    """Three consecutive BasicMAC.select_actions steps with the epsilon-draws injected, against orc.mac_select_actions.
    Q and hidden state within the tier's tolerance (fp32 1e-5, bf16 1e-2).  The actions drawn at random are always equal;
    the greedy ones wherever the oracle's gap between its best and second-best available Q exceeds twice the tolerance
    times max|Q|.  On the fp32 tier that leaves out only near-ties at float rounding (the 27m_vs_30m case has one greedy
    gap of 1.3e-7 max|Q| at t = 0, a tie the GPU's fp32 Q cannot resolve against the float64 oracle)."""
    from cuda_utils import to_batch
    from pymarl_b200 import mac_REGISTRY
    from pymarl_b200.synthetic import make_scheme
    shape_key, over, envs = ROLLOUT_CASES[case]
    shape = _shape(shape_key)
    N, A = shape.n_agents, shape.n_actions
    args = default_args(shape, device="cuda", precision=precision, **over)
    H = args.rnn_hidden_dim
    scheme, groups = make_scheme(shape)
    mac = mac_REGISTRY["basic_mac"](scheme, groups, args)
    mac.cuda()
    rng = np.random.default_rng(6)
    d_in = shape.obs_dim + (A if args.obs_last_action else 0) + (N if args.obs_agent_id else 0)
    agent = orc.init_params(orc.agent_param_shapes(d_in, H, A), rng)
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
        a_ref, q_ref, h = orc.mac_select_actions(p64, fields, t, h, eps, u, expo.reshape(envs, N, A),
                                                 args.obs_last_action, args.obs_agent_id)
        q = seen[-1].cpu().numpy().reshape(q_ref.shape)
        hid = mac.hidden_states.detach().cpu().numpy().reshape(h.shape)
        print(case, precision, t, "q %.1e hidden %.1e" % (rel_err(q, q_ref), rel_err(hid, h)))
        assert rel_err(q, q_ref) < tol, (t, rel_err(q, q_ref))
        assert rel_err(hid, h) < tol, (t, rel_err(hid, h))
        random = u < np.float32(eps)
        avail = fields["avail_actions"][:, t]
        top2 = np.sort(np.where(avail == 0, -np.inf, q_ref), axis=2)[..., -2:]
        gap = top2[..., 1] - top2[..., 0]                   # inf where one action is available
        clear = gap > 2 * tol * np.abs(q_ref).max()
        assert random.any() and (~random & clear).mean() > 0.5 * (~random).mean(), t
        np.testing.assert_array_equal(acts[random], a_ref[random])
        np.testing.assert_array_equal(acts[~random & clear], a_ref[~random & clear])
