"""GPU parity tests of the COMA path (SURVEY.md section 8f rank 4) through the Python mirror and the C ABI: golden fixture
produced by the reference's COMALearner (tests/golden/coma_tiny.npz) and the numpy oracle (oracle/coma_oracle.py, pinned to
the same fixture) run in float64 on SMAC-shaped batches.

The COMA kernels branch on the shape; every branch has a case here that asserts it takes it (see `reaches`):
  - more than 32 actions: the second action per lane (a = lane + 32) of coma_policy_kernel and policy_head_kernel;
  - the target critic pass over T in chunks of nt timesteps (coma_plan), in the train step and in COMACritic.forward;
  - the grid-stride loops of coma_critic_td_kernel, coma_policy_kernel and policy_head_kernel, whose grids are capped.
fp32 tier bounds: see TRAIN_BOUNDS; sampled actions bit-exact given the generator's draws, except on near-ties."""
import copy
import ctypes as C

import numpy as np
import pytest
import torch as th

from golden_utils import Golden, rel_err
from oracle import coma_oracle as co, qlearner_oracle as orc
from pymarl_b200 import _lib
from pymarl_b200.synthetic import SMAC_SHAPES, SmacShape, default_args, numpy_episode_fields, make_scheme, get_shape

gpu = pytest.mark.gpu
TOL = 1e-5
COMA_KW = dict(agent_output_type="pi_logits", action_selector="multinomial", learner="coma_learner", critic_lr=5e-4,
               td_lambda=0.8, mask_before_softmax=True, epsilon_start=0.5, epsilon_finish=0.01, epsilon_anneal_time=100000,
               learner_log_interval=0, test_greedy=True)
TINY = SmacShape("tiny", 2, 4, 4, 3, 5)


def target_chunks(shape, B, T):
    """coma_plan (api.cu): the target critic runs over nt = (64 << 20) / (B*N*D) timesteps per chunk, clamped to [1, T]."""
    s = get_shape(shape)
    D = s.state_dim + s.obs_dim + 2 * s.n_agents * s.n_actions + s.n_agents
    nt = min(max((64 << 20) // (B * s.n_agents * D), 1), T)
    return [min(nt, T - t0) for t0 in range(0, T, nt)]


def grid_of(items, per_block, blocks_per_sm, sms):
    """coma.cu launchers: grid = min(ceil(items / per_block), blocks_per_sm * SMs) -> (blocks, passes of the stride loop)."""
    grid = min(-(-items // per_block), blocks_per_sm * sms)
    return grid, -(-items // (grid * per_block))


def reaches(shape, B, T, sms):
    """The shape-dependent branches a COMA train step at (shape, B, T) takes on a device with `sms` SMs."""
    s = get_shape(shape)
    R = B * s.n_agents
    out = set()
    if s.n_actions > 32:
        out.add("A>32")
    chunks = target_chunks(s, B, T)
    if len(chunks) > 1:
        out.add("chunks " + "+".join(map(str, chunks)))
    if chunks[0] == 1:
        out.add("nt=1")
    blocks, passes = grid_of(R, 256, 4, sms)                 # coma_critic_td_kernel: 256 rows a block, <= 4 * SMs blocks
    if blocks > 1:
        out.add("td blocks %d" % blocks)
    if passes > 1:
        out.add("td loop")
    if grid_of((T - 1) * R, 8, 8, sms)[1] > 1:                # coma_policy_kernel: 8 warps a block, <= 8 * SMs blocks
        out.add("policy loop")
    return out


def build_coma(shape, args, agent=None, critic=None, target_critic=None):
    from cuda_utils import Logger
    from pymarl_b200 import le_REGISTRY, mac_REGISTRY
    shape = get_shape(shape)
    scheme, groups = make_scheme(shape)
    scheme["actions_onehot"] = {"vshape": (shape.n_actions,), "dtype": th.float32, "group": "agents"}
    args.device, args.use_cuda = "cuda", True
    mac = mac_REGISTRY[args.mac](copy.deepcopy(scheme), groups, args)
    logger = Logger()
    learner = le_REGISTRY["coma_learner"](mac, scheme, logger, args)
    learner.cuda()
    ld = lambda m, p: m.load_state_dict({k: th.from_numpy(np.asarray(v, np.float32)) for k, v in p.items()}) if p else None
    ld(mac.agent, agent)
    ld(learner.critic, critic)
    ld(learner.target_critic, target_critic if target_critic is not None else critic)
    return learner, logger


def state_np(m):
    return {k: v.detach().cpu().numpy() for k, v in m.state_dict().items()}


@gpu
def test_coma_golden_forward_pieces_and_action_selection():
    from cuda_utils import to_batch
    g = Golden("coma_tiny")
    args = default_args(g.shape, mixer=None, **g.meta["over"])
    learner, _ = build_coma(g.shape, args, g.group("init/agent"), g.group("init/critic"), g.group("init/target_critic"))
    f = g.batch_fields()
    batch = to_batch(g.shape, f)
    B, T = batch.batch_size, batch.max_seq_length
    # COMACritic.forward: all timesteps and a single one
    tq = learner.target_critic(batch)
    assert rel_err(tq.cpu().numpy(), g["fw/target_q"]) < TOL
    q3 = learner.target_critic(batch, t=3)
    assert q3.shape == (B, 1, g.shape.n_agents, g.shape.n_actions)
    assert rel_err(q3.cpu().numpy()[:, 0], g["fw/target_q"][:, 3]) < TOL
    # BasicMAC.forward with agent_output_type = pi_logits: masked softmax + epsilon floor; plain softmax in test mode
    mac = learner.mac
    assert mac.action_selector.epsilon == float(g["epsilon"])
    mac.init_hidden(B)
    for t in range(T - 1):
        pi = mac.forward(batch, t)
        assert rel_err(pi.cpu().numpy(), g["fw/pi"][:, t]) < TOL, t
    mac.init_hidden(B)
    assert rel_err(mac.forward(batch, 0, test_mode=True).cpu().numpy(), g["fw/pi_test_t0"]) < TOL
    # MultinomialActionSelector: the generator's exponential draws injected -> bit-exact actions; greedy in test mode
    expo = th.from_numpy(g["sel/expo"]).cuda().reshape(-1, g.shape.n_actions).contiguous()
    mac.action_selector.draw = lambda x: expo
    mac.init_hidden(B)
    acts = mac.select_actions(batch, t_ep=0, t_env=1234)
    np.testing.assert_array_equal(acts.cpu().numpy(), g["sel/actions"])
    assert mac.action_selector.epsilon == float(g["sel/epsilon"])
    mac.init_hidden(B)
    np.testing.assert_array_equal(mac.select_actions(batch, t_ep=0, t_env=1234, test_mode=True).cpu().numpy(), g["sel/greedy"])
    # the kernel's own generator: only available actions, roughly the policy's frequencies
    del mac.action_selector.draw
    mac.action_selector.rng = "philox"
    # (A = 36: most of the mass on actions >= 32, the second action of a lane in the kernels with two per lane)
    p36 = np.zeros(36, np.float32)
    p36[[3, 32, 34, 35]] = [0.1, 0.15, 0.45, 0.3]
    for p in (np.array([0.1, 0.0, 0.6, 0.3, 0.0], np.float32), p36):
        A = len(p)
        probs = th.from_numpy(p).cuda().repeat(20000, 1).view(20000, 1, A)
        avail = (probs > 0).int()
        a = mac.action_selector.select_action(probs, avail, 0)
        freq = (th.bincount(a.flatten(), minlength=A).float() / 20000).cpu().numpy()
        assert (freq[p == 0] == 0).all() and (np.abs(freq - p) < 0.02).all(), (A, freq)


@gpu
def test_coma_train_steps_match_reference_golden():
    from cuda_utils import to_batch
    g = Golden("coma_tiny")
    args = default_args(g.shape, mixer=None, **g.meta["over"])
    learner, logger = build_coma(g.shape, args, g.group("init/agent"), g.group("init/critic"), g.group("init/target_critic"))
    batch = to_batch(g.shape, g.batch_fields())
    learner.mac.action_selector.epsilon = float(g["epsilon"])
    for step in range(g.meta["n_steps"]):
        learner.train(batch, step, 0)
        if step == 0:
            ws = learner.workspace_views()
            assert rel_err(ws["targets"].cpu().numpy(), g["fw/td_lambda_targets"]) < TOL
        for k in ("critic_loss", "critic_grad_norm", "td_error_abs", "q_taken_mean", "target_mean", "advantage_mean",
                  "coma_loss", "agent_grad_norm", "pi_max"):
            r = float(g["step%d/stat/%s" % (step, k)])
            assert abs(logger.stats[k][-1][1] - r) <= 3 * TOL * max(1.0, abs(r)), (step, k, logger.stats[k][-1][1], r)
        for tag, mod in (("agent", learner.mac.agent), ("critic", learner.critic), ("target_critic", learner.target_critic)):
            for k, v in g.group("step%d/%s" % (step, tag)).items():
                assert rel_err(state_np(mod)[k], v) < 5 * TOL, (step, tag, k)
        assert learner.critic_training_steps == int(g["step%d/critic_training_steps" % step])
        for tag, opt in (("agent", learner.agent_optimiser), ("critic", learner.critic_optimiser)):
            sq = np.concatenate([s.cpu().numpy().ravel() for s in opt.square_avg])
            assert rel_err(sq, g["step%d/sq/%s" % (step, tag)]) < 1e-4, (step, tag)
    assert logger.infos.count("Updated target network") >= 1


# Bounds for a critic ReLU decision that flips between the fp32 step and the float64 oracle (see the test's docstring).
# One flip, from RMSprop state 1e-2: any single flip in 27m_vs_30m B = 64, T = 16 leaves at most q 6.1e-6, critic step
# stats 5.5e-5, critic parameters 5.9e-5 in the float64 oracle; the B200 shows q 6.0e-6, 5.5e-5, 1.0e-5.
ONE_FLIP = {"q": 3e-5, "stat": 3e-4, "param.critic": 3e-4}
# One flip chained through the 116 critic updates after it: q 1.2e-4, stats 1.4e-3, critic parameters 5.8e-4 on a B200.
FLIP_CHAINED = {"q": 1e-3, "stat": 1e-2, "param.critic": 5e-3}
# shape, B (None: past coma_critic_td_kernel's grid on this device), T, RMSprop state at the start, the branches the case
# is there for (each must be in `reaches`), whether avail_actions is edited (_edit_avail), bounds that replace TRAIN_BOUNDS'
TRAIN_CASES = [
    pytest.param("3m", 16, 20, 0.0, (), False, {}, id="3m-16-20"),
    pytest.param("2s3z", 8, 12, 0.0, (), False, {}, id="2s3z-8-12"),
    pytest.param("MMM2", 6, 8, 0.0, (), False, {}, id="MMM2-6-8"),
    # the only SMAC map with A > 32, at the reference's COMA batch: a ragged last chunk of the target pass
    pytest.param("27m_vs_30m", 8, 120, 1e-2, ("A>32", "chunks 90+30"), False, FLIP_CHAINED, id="27m_vs_30m-8-120"),
    pytest.param("27m_vs_30m", 64, 16, 1e-2, ("A>32", "chunks 11+5", "policy loop", "td blocks 7"), False, ONE_FLIP,
                 id="27m_vs_30m-64-16"),
    pytest.param("27m_vs_30m", 384, 5, 1e-2, ("A>32", "nt=1"), False, {}, id="27m_vs_30m-384-5"),
    # bench.py's coma_record: 119 chained critic updates, each on the critic the previous one left
    pytest.param("2s3z", 8, 120, 1e-2, (), False, {}, id="2s3z-8-120"),
    pytest.param(TINY, None, 5, 1e-2, ("td loop",), False, {}, id="tiny-td_loop-5"),
    pytest.param("27m_vs_30m", 8, 20, 0.0, ("A>32",), True, {}, id="27m_vs_30m-8-20-upper_avail"),
]
# norm-wise relative error bounds, about 10x the largest error observed on a B200 over the cases above
TRAIN_BOUNDS = {"q": 1e-5, "target_q": 1e-5, "targets": 1e-5, "pi": 1e-5, "stat": 3e-5, "agent_stat": 3e-5,
                "param.agent": 5e-5, "param.critic": 5e-5}


def _edit_avail(fields, shape, rng):
    """A quarter of the filled agent-steps may only take actions 32..A-1 (action 0 cleared), a tenth has one legal action
    (mostly >= 32); the taken action is redrawn among the legal ones and the one-hot re-derived."""
    A = shape.n_actions
    av, act = fields["avail_actions"], fields["actions"][..., 0]
    live = np.broadcast_to(fields["filled"][:, :, :1] != 0, act.shape)
    pick = rng.random(act.shape)
    upper, single = live & (pick < 0.25), live & (pick >= 0.25) & (pick < 0.35)
    av[upper | single] = 0
    n_up = int(upper.sum())
    av[upper, 32:] = rng.random((n_up, A - 32)) < 0.5
    av[upper, 32 + rng.integers(0, A - 32, n_up)] = 1
    one = np.where(rng.random(int(single.sum())) < 0.7, rng.integers(32, A, int(single.sum())),
                   rng.integers(0, 32, int(single.sum())))
    av[single, one] = 1
    edited = upper | single
    act[edited] = (rng.random((int(edited.sum()), A)) * av[edited]).argmax(-1)
    oh = np.zeros_like(fields["actions_onehot"])
    np.put_along_axis(oh, act[..., None], 1.0, axis=-1)
    fields["actions_onehot"][...] = oh * fields["filled"][:, :, :, None]
    assert (act[upper] >= 32).all() and (av[single].sum(-1) == 1).all()


@gpu
@pytest.mark.parametrize("shape_name,B,T,sq0,claims,avail_edit,loose", TRAIN_CASES)
def test_coma_train_step_matches_oracle(shape_name, B, T, sq0, claims, avail_edit, loose):
    """One COMALearner.train on a ragged batch (the last three timesteps padding for every episode -> skipped critic
    steps) against the float64 oracle: q_vals (each timestep as scored by the critic of that moment), td-lambda targets,
    the renormalised policy, the stats row of every critic step and of the agent, the logged means, the post-update
    agent and critic parameters, critic_training_steps; and the target critic's COMACritic.forward over all timesteps and
    at one timestep of the last chunk.

    Bounds (TRAIN_BOUNDS) are norm-wise relative (max |err| / max |ref|), stats relative to max(1, |ref|).  The fp32
    step's only discontinuities are the critic's two ReLU masks.  A pre-activation within rounding of zero takes one side
    in fp32 and the other in float64, and the critic updates after it carry the difference: from RMSprop state 0 the
    first updates are lr * sign(g) on the one-hot input columns that only a few rows touch, so a single flip moves such a
    weight by a whole step (27m_vs_30m B = 64, T = 16 from zero state: critic fc1 1.7e-1, q 6e-2).  The same numbers
    come out of the numpy oracle run in float32; with its ReLU decisions pinned into the float64 oracle they fall to
    1.4e-6.  So the 27m cases start from RMSprop state 1e-2 on both sides, which keeps each update close to linear in
    its gradient.  What one flip still leaves there is measured by flipping the pre-activation nearest zero of each
    critic step in the float64 oracle, one at a time: in 27m_vs_30m B = 64, T = 16 the one at t = 8 (|pre| 2e-7) gives q
    6.1e-6, critic grad norm 5.5e-5, critic parameters 9.3e-6, what the B200 shows (ONE_FLIP).  27m_vs_30m T = 120
    chains a flip (at t = 45 in the float32 oracle) through 45 more updates (FLIP_CHAINED).  Only q, the critic step
    stats and the critic parameters get these bounds; targets, the target critic's Q, the policy, the agent's stats and
    parameters keep the tight ones in every case."""
    from cuda_utils import to_batch
    shape = get_shape(shape_name)
    N, A = shape.n_agents, shape.n_actions
    sms = th.cuda.get_device_properties(0).multi_processor_count
    if B is None:
        B = 4 * sms * 256 // N + 64
    assert set(claims) <= reaches(shape, B, T, sms), (claims, reaches(shape, B, T, sms))
    args = default_args(shape, mixer=None, **COMA_KW)
    rng = np.random.default_rng(5)
    agent = orc.init_params(orc.agent_param_shapes(shape.obs_dim + A + N, 64, A), rng)
    crit = co.init_critic(co.critic_param_shapes(shape.state_dim, shape.obs_dim, N, A), rng)
    tcrit = {k: (v + 0.05 * rng.standard_normal(v.shape)).astype(np.float32) for k, v in crit.items()}
    fields = numpy_episode_fields(shape, B, T, seed=17, ragged=True)
    if avail_edit:
        _edit_avail(fields, shape, rng)
    for k in fields:                                       # make the last timesteps padding for every episode
        fields[k][:, T - 3:] = 0
    f64 = lambda p: {k: v.astype(np.float64) for k, v in p.items()}
    olr = co.OracleCOMALearner(f64(agent), f64(crit), copy.copy(args))
    olr.target_critic = f64(tcrit)
    for sq in list(olr.sq_agent.values()) + list(olr.sq_critic.values()):
        sq[...] = sq0
    learner, logger = build_coma(shape, args, agent, crit, tcrit)
    learner._flat["asq"].fill_(sq0)
    learner._flat["csq"].fill_(sq0)
    eps = 0.37
    learner.mac.action_selector.epsilon = eps
    st, _, fw = olr.train(fields, 0, 0, float(np.float32(eps)))
    batch = to_batch(shape, fields)
    learner.train(batch, 0, 0)
    ws = learner.workspace_views()
    mask = fields["filled"][:, :-1, 0].astype(np.float64)
    mask[:, 1:] *= 1 - fields["terminated"][:, :-2, 0]
    live_t = mask.sum(0) > 0                               # q_vals of skipped critic steps stay 0 in the reference
    err = {"targets": rel_err(ws["targets"].cpu().numpy(), fw["targets"]),
           "q": rel_err(ws["q_vals"].cpu().numpy()[:, live_t], fw["q_vals"][:, live_t]),
           "pi": rel_err(ws["pi"].view(T - 1, B, N, A).permute(1, 0, 2, 3).cpu().numpy(), fw["pi"])}
    # COMACritic.forward: all timesteps (chunked like the target pass) and one timestep of the last chunk
    t1 = T - target_chunks(shape, B, T)[-1] // 2 - 1
    err["target_q"] = max(rel_err(learner.target_critic(batch).cpu().numpy(), fw["target_q"]),
                          rel_err(learner.target_critic(batch, t=t1)[:, 0].cpu().numpy(), fw["target_q"][:, t1]))
    # stats rows: critic step t -> [mask_sum, td^2, |td|, q_taken, target sums, grad norm]; row T-1: the agent's
    rows = learner.last_stats.numpy()
    log = fw["critic_log"]
    ts = np.array(log["t"])
    assert sorted(np.nonzero(rows[:T - 1, 0])[0]) == sorted(ts) and (rows[ts, 0] == mask[:, ts].sum(0) * N).all()
    c = rows[ts]
    rel = lambda got, ref: float(np.max(np.abs(np.asarray(got) - ref) / np.maximum(1.0, np.abs(ref))))
    for k, i in (("critic_loss", 1), ("td_error_abs", 2), ("q_taken_mean", 3), ("target_mean", 4)):
        err["stat." + k] = rel(c[:, i] / c[:, 0], np.array(log[k]))
    err["stat.critic_grad_norm"] = rel(c[:, 5], np.array(log["critic_grad_norm"]))
    ag = rows[T - 1]
    assert ag[0] == mask.sum() * N
    for k, v in (("coma_loss", -ag[1] / ag[0]), ("advantage_mean", ag[2] / ag[0]), ("pi_max", ag[3] / ag[0]),
                 ("agent_grad_norm", ag[5])):
        err["agent_stat." + k] = rel(v, st[k])
    for k in ("critic_loss", "critic_grad_norm", "td_error_abs", "q_taken_mean", "target_mean", "advantage_mean",
              "coma_loss", "agent_grad_norm", "pi_max"):
        err["stat.logged." + k] = rel(logger.stats[k][-1][1], st[k])
    assert learner.critic_training_steps == olr.critic_training_steps < T - 1
    for tag, mod, ref in (("agent", learner.mac.agent, olr.agent), ("critic", learner.critic, olr.critic)):
        got = state_np(mod)
        for k, v in ref.items():
            err["param.%s.%s" % (tag, k)] = rel_err(got[k], v)
    print(shape.name, B, T, {k: "%.1e" % v for k, v in err.items()})
    bounds = dict(TRAIN_BOUNDS, **loose)
    for k, e in err.items():
        group = k.split(".")[0] if not k.startswith("param.") else ".".join(k.split(".")[:2])
        assert e < bounds[group], (k, e)


@gpu
def test_coma_checkpoint_round_trip(tmp_path):
    from cuda_utils import to_batch
    shape = SMAC_SHAPES["3m"]
    args = default_args(shape, mixer=None, **COMA_KW)
    fields = numpy_episode_fields(shape, 8, 10, seed=2, ragged=True)
    batch = to_batch(shape, fields)
    a, _ = build_coma(shape, copy.copy(args))
    a.train(batch, 0, 0)
    a.save_models(str(tmp_path))
    import os
    assert sorted(os.listdir(str(tmp_path))) == ["agent.th", "agent_opt.th", "critic.th", "critic_opt.th"]
    b, _ = build_coma(shape, copy.copy(args))
    b.load_models(str(tmp_path))
    a.target_critic.load_state_dict(a.critic.state_dict())           # what load_models does on the other side
    a.train(batch, 1, 0)
    b.train(batch, 1, 0)
    for m1, m2 in ((a.mac.agent, b.mac.agent), (a.critic, b.critic)):
        for k, v in m1.state_dict().items():
            assert th.equal(v, m2.state_dict()[k]), k


def _graph_matches_eager(shape_name, B, T):
    """args.cuda_graph: the ~14 launches per timestep of a COMA step replayed as one graph give the bits of the eager step."""
    from cuda_utils import to_batch
    shape = SMAC_SHAPES[shape_name]
    N, A = shape.n_agents, shape.n_actions
    fields = numpy_episode_fields(shape, B, T, seed=6, ragged=True)
    rng = np.random.default_rng(9)
    agent = orc.init_params(orc.agent_param_shapes(shape.obs_dim + A + N, 64, A), rng)
    crit = co.init_critic(co.critic_param_shapes(shape.state_dim, shape.obs_dim, N, A), rng)
    outs = []
    for graph in (False, True):
        args = default_args(shape, mixer=None, cuda_graph=graph, **COMA_KW)
        lr, _ = build_coma(shape, args, agent, crit, crit)
        batch = to_batch(shape, fields)
        for i in range(4):
            lr.train(batch, i, 0)
        if graph:
            assert any(isinstance(v, tuple) for v in lr._graphs.values())
        outs.append((lr._flat["ap"].clone(), lr._flat["cp"].clone(), lr._flat["tp"].clone(), lr.last_stats.clone()))
    for x, y in zip(*outs):
        assert th.equal(x, y)


@gpu
def test_coma_cuda_graph_step_is_bit_identical():
    _graph_matches_eager("3m", 8, 16)


@gpu
def test_coma_cuda_graph_step_with_chunked_target_pass_is_bit_identical():
    """27m_vs_30m, B = 8, T = 120: the captured graph holds the target pass's chunk loop (90 + 30 timesteps)."""
    assert target_chunks("27m_vs_30m", 8, 120) == [90, 30]
    _graph_matches_eager("27m_vs_30m", 8, 120)


def test_coma_action_limit_is_64():
    """Host only: the COMA kernels hold at most two actions per lane of a warp, so A = 65 is refused before any launch."""
    L = _lib.lib()
    dummy = C.c_void_p(256)                                  # never dereferenced: rows = 0
    for A, ok in ((64, True), (65, False)):
        d = _lib.make_dims(B=8, T=10, N=3, O=30, S=48, A=A, H=64, E=128, mixer=None)
        ws = L.pmb_coma_workspace_bytes(C.byref(d))
        assert (ws > 0) if ok else (ws == -1), (A, ws)
        rc = L.pmb_policy_head(0, A, C.c_float(0.1), 0, dummy, dummy, dummy, None)
        assert (rc == 0) == ok, (A, rc)


def _top2_gap(keys):
    """(best - second best) / best per row; keys -inf where excluded."""
    top2 = np.sort(keys, axis=-1)[..., -2:]
    with np.errstate(invalid="ignore"):
        return (top2[..., 1] - top2[..., 0]) / top2[..., 1]


@gpu
@pytest.mark.parametrize("A", [33, 36, 64])
def test_policy_head_and_multinomial_match_reference(A):
    """pmb_policy_head against co.policy_head in float64 and pmb_multinomial with injected Exp(1) draws against
    co.multinomial_select, on more rows than one pass of policy_head_kernel's grid (8 * SMs blocks of 8 warps, one row
    a warp): rows with no legal action, one legal action, legal actions only at >= 32.  Probabilities within 1e-6 of
    the row's largest; actions equal except on rows whose two best keys differ by less than 2e-6 relative."""
    sms = th.cuda.get_device_properties(0).multi_processor_count
    rows = 3 * 64 * sms + 37
    assert grid_of(rows, 8, 8, sms)[1] > 1
    rng = np.random.default_rng(A)
    logits = (3 * rng.standard_normal((rows, A))).astype(np.float32)
    avail = (rng.random((rows, A)) < 0.5).astype(np.int32)
    avail[:, 0] = 1
    kind = np.arange(rows) % 6
    avail[kind == 1] = 0                                     # no legal action
    for k, lo in ((2, 0), (3, 32)):                          # one legal action anywhere / at >= 32
        n = int((kind == k).sum())
        avail[kind == k] = 0
        avail[np.nonzero(kind == k)[0], rng.integers(lo, A, n)] = 1
    upper = kind == 4                                        # several legal actions, all at >= 32
    avail[upper, :32] = 0
    avail[np.nonzero(upper)[0], rng.integers(32, A, int(upper.sum()))] = 1
    dev = th.device("cuda")
    lg, av = th.from_numpy(logits).to(dev), th.from_numpy(avail).to(dev)
    legal = avail.sum(1) > 0
    s = _lib.stream_ptr(dev)
    for eps, test_mode in ((0.0, False), (0.3, False), (1.0, False), (0.3, True)):
        probs = th.empty_like(lg)
        _lib.check(_lib.lib().pmb_policy_head(rows, A, C.c_float(eps), int(test_mode), _lib.ptr(lg), _lib.ptr(av),
                                              _lib.ptr(probs), s), "pmb_policy_head")
        p = probs.cpu().numpy()
        ref = co.policy_head(logits.astype(np.float64), avail, float(np.float32(eps)), test_mode)
        den = ref.max(1, keepdims=True)
        perr = float((np.abs(p - ref) / np.where(den > 0, den, 1.0)).max())
        expo = rng.exponential(size=(rows, A)).astype(np.float32)
        out = th.empty(rows, dtype=th.int64, device=dev)
        _lib.check(_lib.lib().pmb_multinomial(rows, A, _lib.ptr(probs), _lib.ptr(av), _lib.ptr(th.from_numpy(expo).to(dev)),
                                              int(test_mode), 0, 0, _lib.ptr(out), s), "pmb_multinomial")
        acts = out.cpu().numpy()
        a_ref = co.multinomial_select(p[:, None], avail[:, None], expo[:, None], test_mode)[:, 0]
        pm = np.where(avail != 0, p.astype(np.float64), 0.0)
        with np.errstate(invalid="ignore", divide="ignore"):
            keys = pm if test_mode else (pm / pm.sum(1, keepdims=True)) / expo
        tie = legal & ~(_top2_gap(np.where(avail != 0, keys, -np.inf)) >= 2e-6)
        tie &= avail.sum(1) > 1
        print(A, eps, test_mode, "probs %.1e, near-ties exempt %d of %d rows" % (perr, int(tie.sum()), rows))
        assert perr < 1e-6, (eps, test_mode, perr)
        assert (avail[legal, acts[legal]] == 1).all()
        np.testing.assert_array_equal(acts[~tie], a_ref[~tie])


@gpu
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_coma_rollout_policy_matches_oracle(precision):
    """Three BasicMAC.select_actions steps of the COMA MAC (pi_logits, multinomial) at 27m_vs_30m (A = 36) with the
    Exp(1) draws injected, on more agent rows than one pass of policy_head_kernel's grid: the policy against the float64
    oracle within the tier's tolerance (fp32 1e-5, bf16 1e-2), the actions equal except on rows whose two best keys p/e
    differ by less than twice that tolerance."""
    from cuda_utils import to_batch
    from pymarl_b200 import mac_REGISTRY
    shape = SMAC_SHAPES["27m_vs_30m"]
    N, A = shape.n_agents, shape.n_actions
    sms = th.cuda.get_device_properties(0).multi_processor_count
    envs = 64 * sms // N + 5
    assert grid_of(envs * N, 8, 8, sms)[1] > 1
    args = default_args(shape, mixer=None, device="cuda", precision=precision, **COMA_KW)
    scheme, groups = make_scheme(shape)
    mac = mac_REGISTRY["basic_mac"](scheme, groups, args)
    mac.cuda()
    rng = np.random.default_rng(8)
    agent = orc.init_params(orc.agent_param_shapes(shape.obs_dim + A + N, args.rnn_hidden_dim, A), rng)
    mac.agent.load_state_dict({k: th.from_numpy(v) for k, v in agent.items()})
    p64 = {k: v.astype(np.float64) for k, v in agent.items()}
    fields = numpy_episode_fields(shape, envs, 5, seed=4, ragged=False)
    batch = to_batch(shape, {k: v for k, v in fields.items() if k != "actions_onehot"})
    sel = mac.action_selector
    seen = []
    select = sel.select_action
    sel.select_action = lambda p, *a, **kw: (seen.append(p.detach().clone()), select(p, *a, **kw))[1]
    mac.init_hidden(envs)
    h = np.zeros((envs * N, args.rnn_hidden_dim))
    tol = 1e-5 if precision == "fp32" else 1e-2
    for t in range(3):
        expo = rng.exponential(size=(envs * N, A)).astype(np.float32)
        sel.draw = lambda x, e=th.from_numpy(expo).cuda(): e
        eps = sel.epsilon                                    # BasicMAC.forward floors with the selector's epsilon so far
        acts = mac.select_actions(batch, t_ep=t, t_env=40000).cpu().numpy()
        logits, h = orc.rnn_agent_forward(p64, orc.build_inputs(fields, t).astype(np.float64), h)
        avail = fields["avail_actions"][:, t]
        p_ref = co.policy_head(logits, avail.reshape(-1, A), float(np.float32(eps))).reshape(envs, N, A)
        p = seen[-1].cpu().numpy()
        a_ref = co.multinomial_select(p_ref, avail, expo.reshape(envs, N, A))
        keys = np.where(avail != 0, p_ref / p_ref.sum(-1, keepdims=True) / expo.reshape(envs, N, A), -np.inf)
        clear = _top2_gap(keys) >= 2 * tol
        print(precision, t, "probs %.1e, near-ties exempt %d of %d rows" % (rel_err(p, p_ref), int((~clear).sum()), envs * N))
        assert rel_err(p, p_ref) < tol, (t, rel_err(p, p_ref))
        assert clear.mean() > 0.5
        np.testing.assert_array_equal(acts[clear], a_ref[clear])
