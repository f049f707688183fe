"""CPU oracle for the COMA learner (SURVEY.md section 8f rank 4)  --  TEST INFRASTRUCTURE, NOT PRODUCT CODE.

A numpy restatement of the reference's COMALearner.train (learners/coma_learner.py:32-148), COMACritic
(modules/critics/coma.py:22-59), build_td_lambda_targets (utils/rl_utils.py:4-15), the policy head of BasicMAC.forward
for agent_output_type == "pi_logits" (controllers/basic_controller.py:51-73) and MultinomialActionSelector
(components/action_selectors.py:9-33), with hand-derived backward passes.  Pinned against the reference itself:
tests/golden/make_golden.py runs the unmodified COMALearner on seeded synthetic batches and commits inputs / outputs as
tests/golden/coma_*.npz; tests/test_oracle_golden.py checks every function here against them.  Only tests/ may import
this module.  Paths cited are relative to /root/reference/src; dtype follows the parameters' dtype.
"""
import numpy as np

from . import qlearner_oracle as orc

CRITIC_PARAM_NAMES = ["fc1.weight", "fc1.bias", "fc2.weight", "fc2.bias", "fc3.weight", "fc3.bias"]
NEG = -1e10                      # basic_controller.py:58


def critic_param_shapes(S, O, N, A, hidden=128):
    """modules/critics/coma.py:17-20,52-59: input = state + obs + 2 * N * A (actions, last actions) + N (agent id)."""
    D = S + O + 2 * N * A + N
    return {"fc1.weight": (hidden, D), "fc1.bias": (hidden,), "fc2.weight": (hidden, hidden), "fc2.bias": (hidden,),
            "fc3.weight": (A, hidden), "fc3.bias": (A,)}


def init_critic(shapes, rng, dtype=np.float32):
    out = {}
    for k, shp in shapes.items():
        fan_in = shapes[k.rsplit(".", 1)[0] + ".weight"][1]
        out[k] = rng.uniform(-1 / np.sqrt(fan_in), 1 / np.sqrt(fan_in), size=shp).astype(dtype)
    return out


def critic_inputs(batch, t=None):
    """modules/critics/coma.py:29-50.  t = None: all timesteps [B, T, N, D]; t int: [B, 1, N, D]."""
    obs = batch["obs"]
    B, T, N = obs.shape[:3]
    oh = batch["actions_onehot"]
    A = oh.shape[-1]
    dt = obs.dtype
    ts = slice(None) if t is None else slice(t, t + 1)
    nt = T if t is None else 1
    state = np.broadcast_to(batch["state"][:, ts, None, :], (B, nt, N, batch["state"].shape[-1]))
    acts = np.broadcast_to(oh[:, ts].reshape(B, nt, 1, N * A), (B, nt, N, N * A))
    agent_mask = np.repeat(1 - np.eye(N, dtype=dt), A, axis=1)                          # [N, N*A]: own block zeroed
    acts = acts * agent_mask[None, None]
    if t is None:
        last = np.concatenate([np.zeros_like(oh[:, 0:1]), oh[:, :-1]], axis=1)
    elif t == 0:
        last = np.zeros_like(oh[:, 0:1])
    else:
        last = oh[:, t - 1:t]
    last = np.broadcast_to(last.reshape(B, nt, 1, N * A), (B, nt, N, N * A))
    eye = np.broadcast_to(np.eye(N, dtype=dt)[None, None], (B, nt, N, N))
    return np.concatenate([state.astype(dt), obs[:, ts], acts.astype(dt), last.astype(dt), eye], axis=-1)


def critic_forward(cp, inputs, cache=None):
    """modules/critics/coma.py:22-27."""
    x1 = np.maximum(inputs @ cp["fc1.weight"].T + cp["fc1.bias"], 0)
    x2 = np.maximum(x1 @ cp["fc2.weight"].T + cp["fc2.bias"], 0)
    q = x2 @ cp["fc3.weight"].T + cp["fc3.bias"]
    if cache is not None:
        cache.update(inputs=inputs, x1=x1, x2=x2)
    return q


def critic_backward(cp, cache, dq):
    """Gradients of the six critic tensors for dq = dL/dq [rows, A] (what loss.backward() does, coma_learner.py:126)."""
    x1, x2, inp = cache["x1"], cache["x2"], cache["inputs"]
    g = {"fc3.weight": dq.T @ x2, "fc3.bias": dq.sum(0)}
    dx2 = (dq @ cp["fc3.weight"]) * (x2 > 0)
    g["fc2.weight"], g["fc2.bias"] = dx2.T @ x1, dx2.sum(0)
    dx1 = (dx2 @ cp["fc2.weight"]) * (x1 > 0)
    g["fc1.weight"], g["fc1.bias"] = dx1.T @ inp, dx1.sum(0)
    return g


def td_lambda_targets(rewards, terminated, mask, target_qs, gamma, td_lambda):
    """utils/rl_utils.py:4-15.  rewards / terminated / mask [B, T-1, 1], target_qs [B, T, N] -> [B, T-1, N]."""
    dt = target_qs.dtype
    ret = np.zeros_like(target_qs)
    ret[:, -1] = target_qs[:, -1] * (1 - terminated.sum(axis=1))
    g, lam = dt.type(gamma), dt.type(td_lambda)
    for t in range(ret.shape[1] - 2, -1, -1):
        ret[:, t] = lam * g * ret[:, t + 1] + mask[:, t] * (rewards[:, t] + (1 - lam) * g * target_qs[:, t + 1] * (1 - terminated[:, t]))
    return ret[:, :-1]


def policy_head(logits, avail, epsilon, test_mode=False):
    """controllers/basic_controller.py:51-73 for agent_output_type == "pi_logits", mask_before_softmax = True.
    logits, avail [R, A] -> probabilities [R, A] (rows with no available action come out all-zero)."""
    z = logits.copy()
    z[avail == 0] = NEG
    z = z - z.max(axis=1, keepdims=True)
    e = np.exp(z)
    s = e / e.sum(axis=1, keepdims=True)
    if test_mode:
        return s
    n_av = avail.sum(axis=1, keepdims=True).astype(logits.dtype)
    with np.errstate(divide="ignore", invalid="ignore"):
        out = (1 - epsilon) * s + np.ones_like(s) * epsilon / n_av
    out[avail == 0] = 0.0
    return out


def multinomial_select(probs, avail, expo, test_mode=False, test_greedy=True):
    """components/action_selectors.py:19-31.  probs [b, N, A]; expo: the Exp(1) draws Categorical.sample() consumes
    (torch.multinomial, one sample: arg-max of probs / expo)."""
    p = probs.copy()
    p[avail == 0] = 0.0
    if test_mode and test_greedy:
        return p.argmax(axis=2)
    with np.errstate(divide="ignore", invalid="ignore"):
        pn = (p / p.sum(-1, keepdims=True)).astype(np.float32)
        return (pn / np.asarray(expo, np.float32)).argmax(axis=2)


class OracleCOMALearner:
    """learners/coma_learner.py:9-148 with explicit state."""

    def __init__(self, agent_params, critic_params, args):
        self.args = args
        self.agent = {k: v.copy() for k, v in agent_params.items()}
        self.critic = {k: v.copy() for k, v in critic_params.items()}
        self.target_critic = {k: v.copy() for k, v in critic_params.items()}
        self.sq_agent = {k: np.zeros_like(v) for k, v in self.agent.items()}
        self.sq_critic = {k: np.zeros_like(v) for k, v in self.critic.items()}
        self.critic_training_steps = 0
        self.last_target_update_step = 0
        self.n_target_updates = 0

    def _train_critic(self, batch, rewards, terminated, actions, mask):
        """coma_learner.py:103-148.  Returns q_vals [B, T-1, N, A] (each timestep with the critic of that moment), the
        per-step logs (log["t"]: the timestep of each entry), the td-lambda targets and the target critic's Q [B, T, N, A]."""
        a = self.args
        B, T, N = batch["obs"].shape[:3]
        dt = self.critic["fc1.weight"].dtype
        tq = critic_forward(self.target_critic, critic_inputs(batch).reshape(B * T * N, -1).astype(dt)).reshape(B, T, N, -1)
        targets_taken = np.take_along_axis(tq, actions, axis=3)[..., 0]
        targets = td_lambda_targets(rewards, terminated, mask, targets_taken, a.gamma, a.td_lambda)
        A = tq.shape[-1]
        q_vals = np.zeros((B, T - 1, N, A), dtype=dt)
        log = {k: [] for k in ("t", "critic_loss", "critic_grad_norm", "td_error_abs", "target_mean", "q_taken_mean")}
        for t in reversed(range(T - 1)):
            mask_t = np.broadcast_to(mask[:, t], (B, N))
            if mask_t.sum() == 0:
                continue
            cache = {}
            q_t = critic_forward(self.critic, critic_inputs(batch, t).reshape(B * N, -1).astype(dt), cache).reshape(B, N, A)
            q_vals[:, t] = q_t
            q_taken = np.take_along_axis(q_t, actions[:, t], axis=2)[..., 0]
            td = q_taken - targets[:, t]
            mtd = td * mask_t
            msum = mask_t.sum(dtype=dt)
            loss = (mtd ** 2).sum(dtype=dt) / msum
            dq = np.zeros((B, N, A), dtype=dt)
            np.put_along_axis(dq, actions[:, t], (2 * mtd * mask_t / msum)[..., None], axis=2)
            grads = critic_backward(self.critic, cache, dq.reshape(B * N, A))
            gn = orc.clip_grad_norm(grads, CRITIC_PARAM_NAMES, a.grad_norm_clip)
            orc.rmsprop_step(self.critic, grads, self.sq_critic, CRITIC_PARAM_NAMES, a.critic_lr, a.optim_alpha, a.optim_eps)
            self.critic_training_steps += 1
            me = float(msum)
            log["t"].append(t)
            log["critic_loss"].append(float(loss)); log["critic_grad_norm"].append(float(gn))
            log["td_error_abs"].append(float(np.abs(mtd).sum()) / me)
            log["q_taken_mean"].append(float((q_taken * mask_t).sum()) / me)
            log["target_mean"].append(float((targets[:, t] * mask_t).sum()) / me)
        return q_vals, log, targets, tq

    def train(self, batch, t_env, episode_num, epsilon):
        """coma_learner.py:32-101.  `epsilon` = mac.action_selector.epsilon at the time of the call (the epsilon floor of
        BasicMAC.forward, basic_controller.py:62-70)."""
        a = self.args
        B, T, N = batch["obs"].shape[:3]
        dt = self.agent["fc1.weight"].dtype
        rewards = batch["reward"][:, :-1].astype(dt)
        actions = batch["actions"]
        terminated = batch["terminated"][:, :-1].astype(dt)
        mask = batch["filled"][:, :-1].astype(dt)
        mask[:, 1:] = mask[:, 1:] * (1 - terminated[:, :-1])
        avail = batch["avail_actions"][:, :-1]
        q_vals, clog, targets, tq = self._train_critic(batch, rewards, terminated, actions, mask)
        actions = actions[:, :-1]
        A = q_vals.shape[-1]
        # agent unroll over t = 0 .. T-2 (coma_learner.py:55-60)
        sub = {k: v[:, :-1] for k, v in batch.items()}
        logits, cache = orc.mac_unroll(self.agent, sub, getattr(a, "obs_last_action", True), getattr(a, "obs_agent_id", True), True)
        R = B * (T - 1) * N
        av = avail.reshape(R, A)
        pi0 = policy_head(logits.reshape(R, A).astype(dt), av, dt.type(epsilon))            # BasicMAC.forward
        p = pi0.copy()
        p[av == 0] = 0                                                                         # :63
        with np.errstate(divide="ignore", invalid="ignore"):
            Z = p.sum(-1, keepdims=True)
            pi = p / Z                                                                         # :64
        pi[av == 0] = 0                                                                        # :65
        qv = q_vals.reshape(R, A)
        baseline = (pi * qv).sum(-1)
        act = actions.reshape(R, 1)
        q_taken = np.take_along_axis(qv, act, axis=1)[:, 0]
        pi_taken = np.take_along_axis(pi, act, axis=1)[:, 0]
        m = np.broadcast_to(mask, (B, T - 1, N)).reshape(R)
        pi_taken = np.where(m == 0, dt.type(1.0), pi_taken)
        log_pi = np.log(pi_taken)
        adv = q_taken - baseline
        msum = m.sum(dtype=dt)
        coma_loss = -((adv * log_pi) * m).sum(dtype=dt) / msum
        # backward: G = dL/dlog(pi_taken); through renormalisation, the epsilon floor and the masked softmax
        G = np.where(m == 0, 0, -adv * m / msum).astype(dt)
        onehot = np.zeros((R, A), dtype=dt)
        np.put_along_axis(onehot, act, 1.0, axis=1)
        with np.errstate(divide="ignore", invalid="ignore"):
            dp = np.where(av != 0, G[:, None] * (onehot / np.where(pi_taken == 0, 1, (pi_taken * Z[:, 0]))[:, None] - 1.0 / Z), 0)
        dp = np.nan_to_num(dp, nan=0.0, posinf=0.0, neginf=0.0)
        ds = (1 - dt.type(epsilon)) * dp                                                       # unavailable entries carry no gradient
        z = logits.reshape(R, A).astype(dt).copy()
        z[av == 0] = NEG
        z = z - z.max(axis=1, keepdims=True)
        e = np.exp(z)
        s = e / e.sum(axis=1, keepdims=True)
        dz = s * (ds - (ds * s).sum(-1, keepdims=True))
        dz[av == 0] = 0
        dq_full = dz.reshape(B, T - 1, N, A)
        grads = agent_bptt_dense(self.agent, cache, dq_full, B, N)
        raw = {k: v.copy() for k, v in grads.items()}
        names = orc.AGENT_PARAM_NAMES
        gn = orc.clip_grad_norm(grads, names, a.grad_norm_clip)
        orc.rmsprop_step(self.agent, grads, self.sq_agent, names, a.lr, a.optim_alpha, a.optim_eps)
        if (self.critic_training_steps - self.last_target_update_step) / a.target_update_interval >= 1.0:
            for k, v in self.critic.items():
                self.target_critic[k][...] = v
            self.last_target_update_step = self.critic_training_steps
            self.n_target_updates += 1
        n_log = max(1, len(clog["critic_loss"]))
        stats = {k: sum(v) / n_log for k, v in clog.items() if k != "t"}
        me = float(msum)
        stats.update(advantage_mean=float((adv * m).sum()) / me, coma_loss=float(coma_loss), agent_grad_norm=float(gn),
                     pi_max=float((pi.max(axis=1) * m).sum()) / me)
        return stats, raw, dict(q_vals=q_vals, pi=pi.reshape(B, T - 1, N, A), targets=targets, advantages=adv.reshape(B, T - 1, N),
                                logits=logits, target_q=tq, critic_log=clog)


def agent_bptt_dense(p, cache, dq_full, B, N):
    """BPTT through the agent unroll for a DENSE dL/d(logits) [B, T', N, A] (qlearner_oracle.agent_bptt is the
    chosen-action special case)."""
    T = len(cache)
    H = p["fc1.weight"].shape[0]
    dt = p["fc1.weight"].dtype
    g = {k: np.zeros_like(v) for k, v in p.items()}
    dh_next = np.zeros((B * N, H), dtype=dt)
    for t in range(T - 1, -1, -1):
        c = cache[t]
        dq = dq_full[:, t].reshape(B * N, -1).astype(dt)
        g["fc2.weight"] += dq.T @ c["h"]
        g["fc2.bias"] += dq.sum(0)
        dh = dh_next + dq @ p["fc2.weight"]
        r, z, n, ghn, h_in = c["r"], c["z"], c["n"], c["ghn"], c["h_in"]
        dn = dh * (1 - z)
        dz = dh * (h_in - n)
        da_n = dn * (1 - n * n)
        da_r = (da_n * ghn) * r * (1 - r)
        da_z = dz * z * (1 - z)
        dgi = np.concatenate([da_r, da_z, da_n], axis=1)
        dgh = np.concatenate([da_r, da_z, da_n * r], axis=1)
        g["rnn.weight_ih"] += dgi.T @ c["x"]
        g["rnn.bias_ih"] += dgi.sum(0)
        g["rnn.weight_hh"] += dgh.T @ h_in
        g["rnn.bias_hh"] += dgh.sum(0)
        dx = dgi @ p["rnn.weight_ih"]
        dh_next = dh * z + dgh @ p["rnn.weight_hh"]
        dpre1 = dx * (c["x"] > 0)
        g["fc1.weight"] += dpre1.T @ c["inputs"]
        g["fc1.bias"] += dpre1.sum(0)
    return g
