"""Parity evidence for the tensor-core (bf16 operand, fp32 accumulate) tier - the tier every bench number comes from.

1. referee: the few-percent error of the fc1 / hypernet weight gradients against the reference algorithm is claimed
   (DESIGN.md section 2) to come from the step's DISCONTINUOUS decisions flipping on bf16-rounded pre-activations (ReLU
   mask after fc1, sign of the |.| on the hypernet outputs, ReLU in V, the double-Q arg-max).  The test reads those
   decisions out of the GPU step (workspace after a forward-only run), applies them inside the float64 oracle, and
   requires every gradient tensor AND every parameter update to agree within 1e-2 - i.e. what remains with the decisions
   pinned is plain rounding; a wrong term in a backward kernel would not fit.
2. updates, not parameters: (p' - p) of the GPU step against (p' - p) of the oracle, per tensor in the relative L2 norm,
   plus the fraction of sign mismatches on the elements whose gradient is well above the noise.
3. bench scale: the bf16 tier at BASELINE config 4 size (27m_vs_30m, B = 4096, T = 180: 864 row tiles, persistent
   multi-wave kernels, split reductions) against the fp32 tier (pinned to the reference at 1e-5) run over the same
   device batch in chunks of episodes (loss sums and un-normalised gradients are additive over episodes); the same for
   the 16384-env rollout step.
4. VDN and IQL on MMM2 shapes at a batch that needs more than one wave of CTAs (320 row tiles on 148 SMs).
5. additivity / padding invariance (the data-parallel invariant) on the bf16 tier.
"""
import copy

import numpy as np
import pytest
import torch as th

from golden_utils import rel_err
from oracle import qlearner_oracle as orc
from pymarl_b200.synthetic import SMAC_SHAPES, numpy_episode_fields, default_args, torch_episode_fields

pytestmark = pytest.mark.gpu
TOL_BF16 = 1e-2


def _l2(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))


def _oracle_learner(shape, args, seed, dtype=np.float32):
    rng = np.random.default_rng(seed)
    d_in = shape.obs_dim + shape.n_actions + shape.n_agents
    agent = orc.init_params(orc.agent_param_shapes(d_in, args.rnn_hidden_dim, shape.n_actions), rng)
    mixer = orc.init_params(orc.qmix_param_shapes(shape.state_dim, shape.n_agents, args.mixing_embed_dim), rng) \
        if args.mixer == "qmix" else {}
    lr = orc.OracleQLearner(agent, mixer, args)
    for k in lr.target_agent:
        lr.target_agent[k] = (lr.target_agent[k] + 0.05 * rng.standard_normal(lr.target_agent[k].shape)).astype(np.float32)
    for k in lr.target_mixer_p:
        lr.target_mixer_p[k] = (lr.target_mixer_p[k] + 0.02 * rng.standard_normal(lr.target_mixer_p[k].shape)).astype(np.float32)
    if dtype != np.float32:
        for d in (lr.agent, lr.mixer_p, lr.target_agent, lr.target_mixer_p, lr.sq_agent, lr.sq_mixer):
            for k in d:
                d[k] = d[k].astype(dtype)
    return lr


@pytest.mark.parametrize("shape_name,B,T,mixer", [("3m", 32, 60, "qmix"), ("2s3z", 40, 30, "qmix"),
                                                   ("MMM2", 16, 20, "vdn"), ("MMM2", 16, 20, None),
                                                   ("27m_vs_30m", 8, 12, "qmix")])
def test_bf16_gradients_and_updates_match_oracle_with_pinned_decisions(shape_name, B, T, mixer):
    from cuda_utils import build_learner, to_batch, gpu_decisions
    shape = SMAC_SHAPES[shape_name]
    args = default_args(shape, mixer=mixer, learner_log_interval=0, precision="bf16", grad_norm_clip=1e30)
    fields = numpy_episode_fields(shape, B, T, seed=31, ragged=True)
    base = _oracle_learner(shape, copy.copy(args), seed=12)
    dec = gpu_decisions(shape, args, base, fields,
                        which=("relu_mask", "cur_max", "hypernet") if mixer == "qmix" else ("relu_mask", "cur_max"))

    def oracle_run(decisions, dtype):
        o = _oracle_learner(shape, copy.copy(args), seed=12, dtype=dtype)
        for sq in list(o.sq_agent.values()) + list(o.sq_mixer.values()):
            sq[...] = 1e-2                       # pre-warmed RMSprop state: the update is ~linear in the gradient
        p0 = {("agent." + k): v.copy() for k, v in o.agent.items()}
        p0.update({("mixer." + k): v.copy() for k, v in o.mixer_p.items()})
        f = {k: (v.astype(dtype) if v.dtype == np.float32 else v) for k, v in fields.items()}
        stats, raw_grads, fw = o.train(f, 0, 0, decisions=decisions)
        p1 = {("agent." + k): v for k, v in o.agent.items()}
        p1.update({("mixer." + k): v for k, v in o.mixer_p.items()})
        return stats, raw_grads, {k: p1[k].astype(np.float64) - p0[k].astype(np.float64) for k in p0}, fw

    stats_ref, g_ref, u_ref, fw_ref = oracle_run(None, np.float32)          # the reference algorithm as is
    stats_pin, g_pin, u_pin, _ = oracle_run(dec, np.float64)                # float64, GPU's decisions pinned

    learner, _ = build_learner(shape, copy.copy(args), base.agent, base.target_agent, base.mixer_p, base.target_mixer_p)
    learner._flat["sq"].fill_(1e-2)
    p0 = learner._flat["p"].clone()
    learner.train(to_batch(shape, fields), 0, 0)
    st = learner.stats()
    named = {("agent." + k): v for k, v in learner.mac.agent.named_parameters()}
    if learner.mixer is not None:
        named.update({("mixer." + k): v for k, v in learner.mixer.named_parameters()})
    base_ptr = learner._flat["p"].data_ptr()
    report = {}
    for k, prm in named.items():
        off = (prm.data_ptr() - base_ptr) // 4
        g_gpu = prm.grad.cpu().numpy().astype(np.float64)
        u_gpu = (prm.detach() - p0[off:off + prm.numel()].view(prm.shape)).double().cpu().numpy()
        # sign agreement of the update on the elements whose reference gradient is well above the noise floor
        big = np.abs(g_ref[k]) > 0.2 * np.abs(g_ref[k]).max()
        flips = float((np.sign(u_gpu[big]) != np.sign(u_ref[k][big])).mean()) if big.any() else 0.0
        report[k] = dict(grad_vs_ref=_l2(g_gpu, g_ref[k]), grad_vs_pinned=_l2(g_gpu, g_pin[k]),
                         upd_vs_ref=_l2(u_gpu, u_ref[k]), upd_vs_pinned=_l2(u_gpu, u_pin[k]), sign_flips=flips)
    print({k: {a: "%.1e" % b for a, b in v.items()} for k, v in report.items()})
    for k, r in report.items():
        # with the decisions pinned: rounding only, every tensor within the tier's 1e-2
        assert r["grad_vs_pinned"] < TOL_BF16, (k, r)
        assert r["upd_vs_pinned"] < TOL_BF16, (k, r)
        # against the unmodified reference algorithm: the tensors behind a discontinuity carry the flip noise
        # (the RMSprop update is a non-linear, element-wise function of the gradient: it roughly doubles the relative error)
        loose = 0.15 if k.startswith("mixer.") else (5e-2 if k.startswith("agent.fc1") else 2e-2)
        assert r["grad_vs_ref"] < loose and r["upd_vs_ref"] < 2 * loose, (k, r)
        assert r["sign_flips"] < 0.01, (k, r)
    for key in ("loss", "grad_norm", "td_error_abs", "q_taken_mean", "target_mean"):
        assert abs(st[key] - stats_ref[key]) <= 2 * TOL_BF16 * max(1.0, abs(stats_ref[key])), (key, st[key], stats_ref[key])
        assert abs(st[key] - stats_pin[key]) <= TOL_BF16 * max(1.0, abs(stats_pin[key])), (key, st[key], stats_pin[key])


@pytest.mark.parametrize("mixer", ["vdn", None])
def test_bf16_mmm2_more_than_one_wave(mixer):
    """VDN and IQL (BASELINE config 3) on MMM2 shapes with 4096 episodes: R = 40960 rows = 320 row tiles, more than one
    wave of the persistent recurrence kernels (2 tiles per CTA on 148 SMs) - statistics, Q and gradients vs the oracle."""
    from cuda_utils import build_learner, to_batch
    shape = SMAC_SHAPES["MMM2"]
    B, T = 4096, 10
    args = default_args(shape, mixer=mixer, learner_log_interval=0, precision="bf16", grad_norm_clip=1e30, keep_q=1)
    fields = numpy_episode_fields(shape, B, T, seed=33, ragged=True)
    olr = _oracle_learner(shape, copy.copy(args), seed=14)
    learner, _ = build_learner(shape, args, olr.agent, olr.target_agent, {}, {})
    stats, raw_grads, fw = olr.train(fields, 0, 0)
    learner.train(to_batch(shape, fields), 0, 0)
    st = learner.stats()
    for key in ("loss", "grad_norm", "td_error_abs", "q_taken_mean", "target_mean"):
        assert abs(st[key] - stats[key]) <= TOL_BF16 * max(1.0, abs(stats[key])), (key, st[key], stats[key])
    ws = learner.workspace_views(learner._last_dims)
    q = ws["q_on"].view(T, B, shape.n_agents, -1).permute(1, 0, 2, 3).cpu().numpy()
    assert rel_err(q, fw["mac_out"]) < TOL_BF16
    assert rel_err(ws["chosen"].cpu().numpy(), fw["chosen"]) < TOL_BF16
    for k, v in raw_grads.items():
        got = dict(learner.mac.agent.named_parameters())[k.split(".", 1)[1]].grad.cpu().numpy()
        assert _l2(got, v) < (5e-2 if "fc1" in k else TOL_BF16), (k, _l2(got, v))


def test_bf16_full_size_additivity_and_padding():
    """test_full_size_properties_27m on the tensor-core tier: loss sums and un-normalised gradients of a batch equal the
    sums over its halves (different tile composition -> fp32 summation order only), all-padding episodes change nothing."""
    from cuda_utils import build_learner, to_batch
    shape = SMAC_SHAPES["27m_vs_30m"]
    B, T = 64, 60
    fields = numpy_episode_fields(shape, B, T, seed=5, ragged=True)
    args = default_args(shape, mixer="qmix", learner_log_interval=0, grad_norm_clip=1e30, precision="bf16")
    olr = _oracle_learner(shape, copy.copy(args), seed=13)

    def run(sub):
        learner, _ = build_learner(shape, copy.copy(args), olr.agent, olr.target_agent, olr.mixer_p, olr.target_mixer_p)
        learner.train(to_batch(shape, sub), 0, 0)
        st = learner.last_stats.clone().cpu().numpy()
        n = learner._flat["layout"].n_total
        return st, learner._flat["g"][:n].clone().double().cpu().numpy() * st[0]
    full_st, full_g = run(fields)
    h1_st, h1_g = run({k: v[:B // 2] for k, v in fields.items()})
    h2_st, h2_g = run({k: v[B // 2:] for k, v in fields.items()})
    for i in range(5):
        assert abs(full_st[i] - (h1_st[i] + h2_st[i])) <= 1e-5 * max(1.0, abs(full_st[i])), i
    assert rel_err(h1_g + h2_g, full_g) < 1e-4
    pad = {k: np.concatenate([v, np.zeros_like(v[:8])], 0) for k, v in fields.items()}
    pad_st, pad_g = run(pad)
    for i in range(5):
        assert abs(full_st[i] - pad_st[i]) <= 1e-6 * max(1.0, abs(full_st[i])), i
    assert rel_err(pad_g, full_g) < 1e-4


def _tensor_slices(learner):
    lay = learner._flat["layout"]
    from pymarl_b200._lib import PARAM_ORDER
    return {PARAM_ORDER[i]: (lay.offset[i], lay.numel[i]) for i in range(len(PARAM_ORDER)) if lay.numel[i]}


def test_bf16_bench_scale_matches_fp32_tier():
    """BASELINE config 4 at FULL size (27m_vs_30m, B = 4096, T = 180) on the bf16 tier - the exact launch bench.py times -
    against the fp32 tier (pinned to the reference at 1e-5 by the golden tests) run over the SAME device batch in chunks
    of 256 episodes: the five loss sums, chosen-Q / Q_tot per episode chunk, and the un-normalised flat gradient."""
    from cuda_utils import Logger
    from pymarl_b200 import le_REGISTRY, mac_REGISTRY
    from pymarl_b200.synthetic import make_scheme
    free, _ = th.cuda.mem_get_info()
    if free < 110e9:
        pytest.skip("needs ~100 GB of HBM")
    shape = SMAC_SHAPES["27m_vs_30m"]
    B, T, chunk = 4096, 180, 256
    dev = th.device("cuda")

    def make(precision):
        args = default_args(shape, mixer="qmix", device="cuda", use_cuda=True, learner_log_interval=10 ** 12,
                            precision=precision, grad_norm_clip=1e30)
        th.manual_seed(7)
        scheme, groups = make_scheme(shape)
        scheme["actions_onehot"] = {"vshape": (shape.n_actions,), "dtype": th.float32, "group": "agents"}
        mac = mac_REGISTRY["basic_mac"](scheme, groups, args)
        lr = le_REGISTRY["q_learner"](mac, scheme, Logger(), args)
        lr.cuda()
        with th.no_grad():                      # targets differ from the online nets
            g = th.Generator(device="cuda").manual_seed(3)
            lr._flat["target"].add_(0.03 * th.randn(lr._flat["target"].shape, generator=g, device="cuda"))
        return lr

    class DB:
        def __init__(self, f, b):
            self.fields, self.batch_size, self.max_seq_length, self.device = f, b, T, dev

        def __getitem__(self, k):
            return self.fields[k]

    fields = torch_episode_fields(shape, B, T, seed=77, ragged=True, device=dev, with_onehot=False)
    lb = make("bf16")
    p0 = lb._flat["p"].clone()
    lb.train(DB(fields, B), 0, 0)
    th.cuda.synchronize()
    n = lb._flat["layout"].n_total
    st_b = lb.last_stats.clone().cpu().numpy()
    g_b = (lb._flat["g"][:n].double() * st_b[0]).cpu().numpy()
    ws = lb.workspace_views(lb._last_dims)
    chosen_b, qtot_b, tmax_b = ws["chosen"].clone(), ws["q_tot"].clone(), ws["tmax"].clone()
    slices = _tensor_slices(lb)
    del ws
    lb._workspace = None
    th.cuda.empty_cache()

    lf = make("fp32")
    st_f, g_f = np.zeros(5), np.zeros(n)
    abs_q = 0.0                                   # sum |q_tot|: the scale of the (cancelling) q_taken / target sums
    worst = dict(chosen=0.0, q_tot=0.0, tmax_mismatch=0.0)
    for b0 in range(0, B, chunk):
        lf._flat["p"].copy_(p0)                                      # same parameters for every chunk
        lf._flat["sq"].zero_()
        sub = {k: v[b0:b0 + chunk] for k, v in fields.items()}
        lf.train(DB(sub, chunk), 0, 0)
        s = lf.last_stats.clone().cpu().numpy()
        st_f += s[:5]
        g_f += (lf._flat["g"][:n].double() * s[0]).cpu().numpy()
        w = lf.workspace_views(lf._last_dims)
        sl = slice(b0, b0 + chunk)
        worst["chosen"] = max(worst["chosen"], float((w["chosen"] - chosen_b[sl]).abs().max() / w["chosen"].abs().max()))
        worst["q_tot"] = max(worst["q_tot"], float((w["q_tot"] - qtot_b[sl]).abs().max() / w["q_tot"].abs().max()))
        bad = ((w["tmax"] - tmax_b[sl]).abs() > 1e-2 * w["tmax"].abs().max()).float().mean().item()
        worst["tmax_mismatch"] = max(worst["tmax_mismatch"], bad)
        abs_q += float(w["q_tot"].abs().sum())
    errs = {k: _l2(g_b[o:o + m], g_f[o:o + m]) for k, (o, m) in slices.items()}
    print("stats bf16", st_b[:5], "fp32", st_f, worst, {k: "%.1e" % v for k, v in errs.items()})
    for i in range(5):
        # sums 3 and 4 (q_taken, targets) add terms of both signs: their error is measured against sum |q_tot|
        scale = max(1.0, abs(st_f[i]), abs_q if i >= 3 else 0.0)
        assert abs(st_b[i] - st_f[i]) <= TOL_BF16 * scale, (i, st_b[i], st_f[i], scale)
    assert worst["chosen"] < TOL_BF16 and worst["q_tot"] < TOL_BF16, worst
    assert worst["tmax_mismatch"] < 0.03, worst           # double-Q arg-max near-ties flip for a small fraction of the entries
    for k, e in errs.items():
        loose = 0.15 if k.startswith("mixer.") else (5e-2 if k.startswith("agent.fc1") else 2e-2)
        assert e < loose, (k, e)


def test_bf16_rollout_at_bench_scale_matches_fp32_tier():
    """BASELINE config 5 size (16384 envs x 27 agents): three consecutive select_actions steps of the tensor-core rollout
    path against the fp32 path on the same batch: Q and hidden state within 1e-2, greedy actions agree except on near-ties."""
    from pymarl_b200 import mac_REGISTRY
    from pymarl_b200.synthetic import make_scheme
    shape = SMAC_SHAPES["27m_vs_30m"]
    envs, dev = 16384, th.device("cuda")
    fields = torch_episode_fields(shape, envs, 4, seed=5, ragged=False, device=dev, with_onehot=False)

    class DB:
        def __init__(self, f):
            self.fields, self.batch_size, self.max_seq_length, self.device = f, envs, 4, dev

        def __getitem__(self, k):
            return self.fields[k]
    batch = DB(fields)
    macs = {}
    for prec in ("fp32", "bf16"):
        args = default_args(shape, device="cuda", precision=prec)
        scheme, groups = make_scheme(shape)
        th.manual_seed(11)
        macs[prec] = mac_REGISTRY["basic_mac"](scheme, groups, args)
        macs[prec].cuda()
        macs[prec].init_hidden(envs)
    macs["bf16"].agent.load_state_dict(macs["fp32"].agent.state_dict())
    for t in range(3):
        qf = macs["fp32"].forward(batch, t)
        qb = macs["bf16"].forward(batch, t)
        assert float((qf - qb).abs().max() / qf.abs().max()) < TOL_BF16, t
        hf, hb = macs["fp32"].hidden_states.view(-1, 64), macs["bf16"].hidden_states.view(-1, 64)
        assert float((hf - hb).abs().max() / hf.abs().max()) < TOL_BF16, t
        avail = fields["avail_actions"][:, t]
        af = qf.masked_fill(avail == 0, -float("inf")).argmax(2)
        ab = qb.masked_fill(avail == 0, -float("inf")).argmax(2)
        assert float((af != ab).float().mean()) < 0.02, t
        assert bool(avail.gather(2, ab[..., None]).all())
