"""The reference COMA learner step, restated as a custom learner, on COMACritic's autograd path (args.autograd_modules)
against the same learner with a plain nn.Linear fp32 critic.

The step is the one tests/test_critic_autograd.py checks against the reference's recorded run: coma_learner.py:37-148
with the target critic over the whole batch under no_grad, td-lambda targets, one critic RMSprop step per timestep
backwards in time, and the actor loss through BasicMAC.forward with pi_logits.  Two arms on the same GPU and the same data,
both with this package's BasicMAC (autograd_modules = True):
  pmb    this package's COMACritic: one autograd node per critic call, pmb_coma_critic_step_fwd / _bwd
  torch  three nn.Linear layers in fp32 on the GPU, the critic input built with torch ops as coma.py:29-50 builds it
Each step is timed with CUDA events; the arms alternate within every round.  The library launches of one critic
forward and backward at a single timestep are counted with pmb_launch_count.  The card name, power limit and SM clock
are read in the same run.

    python tools/critic_autograd_bench.py --steps 5 --warmup 2 --out profiles/r06_critic_autograd.json
"""
import argparse
import json
import os
import sys

import numpy as np
import torch as th

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.join(REPO, "tests"))
sys.path.insert(0, os.path.join(REPO, "tools"))

from autograd_bench import _gpu_info  # noqa: E402
from cuda_utils import to_batch  # noqa: E402
from test_coma_gpu import COMA_KW  # noqa: E402
from test_critic_autograd import CustomCOMALearner, RefCritic, package_learner, ref_critic_inputs  # noqa: E402
from pymarl_b200 import _lib, mac_REGISTRY  # noqa: E402
from pymarl_b200.synthetic import SMAC_SHAPES, default_args, make_scheme, numpy_episode_fields  # noqa: E402

# the reference's on-policy COMA batch (batch_size_run 8 episodes of up to 120 steps)
CONFIGS = [("2s3z", 8, 120), ("27m_vs_30m", 8, 120)]


class TorchCritic(RefCritic):
    """COMACritic.forward(batch, t) on plain torch: the input built per call (coma.py:29-50), three nn.Linear layers."""

    def __init__(self, shape):
        D = shape.state_dim + shape.obs_dim + 2 * shape.n_agents * shape.n_actions + shape.n_agents
        super().__init__(D, shape.n_actions)
        self.N, self.A = shape.n_agents, shape.n_actions

    def forward(self, batch, t=None):
        f = {k: batch[k] for k in ("state", "obs", "actions_onehot")}
        return super().forward(ref_critic_inputs(f, t, self.N, self.A))[0]


def critic_launches(critic, batch):
    L = _lib.lib()
    th.cuda.synchronize()
    n0 = L.pmb_launch_count()
    q = critic(batch, 5)
    n1 = L.pmb_launch_count()
    q.sum().backward()
    n2 = L.pmb_launch_count()
    for p in critic.parameters():
        p.grad = None
    return n1 - n0, n2 - n1


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    assert th.cuda.is_available(), "critic_autograd_bench needs a CUDA device"
    record = {"what": "custom COMA learner step (coma_learner.py:37-148 on BasicMAC + a critic, torch RMSprop), ragged "
                      "episodes; median ms per step over --steps CUDA-event-timed steps per round, arms alternated",
              "steps": a.steps, "warmup": a.warmup, "rounds": a.rounds, "gpu": _gpu_info(), "configs": {}}
    for shape_key, B, T in CONFIGS:
        shape = SMAC_SHAPES[shape_key]
        args = default_args(shape, mixer=None, **dict(COMA_KW, autograd_modules=True, device="cuda", use_cuda=True))
        fields = numpy_episode_fields(shape, B, T, seed=1, ragged=True)
        batch = to_batch(shape, fields)
        pmb = package_learner(shape, args)
        scheme, groups = make_scheme(shape)
        mac = mac_REGISTRY[args.mac](scheme, groups, args)
        mac.cuda()
        mac.agent.load_state_dict(pmb.mac.agent.state_dict())
        critic = TorchCritic(shape).cuda()
        critic.load_state_dict(pmb.critic.state_dict())
        arms = {"pmb": pmb, "torch": CustomCOMALearner(mac, critic, args)}
        for learner in arms.values():
            learner.mac.action_selector.epsilon = 0.1
            for _ in range(a.warmup):
                learner.train(batch)
        th.cuda.synchronize()
        ms = {arm: [] for arm in arms}
        for _ in range(a.rounds):
            for arm, learner in arms.items():
                times = []
                for _ in range(a.steps):
                    e0, e1 = th.cuda.Event(enable_timing=True), th.cuda.Event(enable_timing=True)
                    e0.record()
                    learner.train(batch)
                    e1.record()
                    e1.synchronize()
                    times.append(e0.elapsed_time(e1))
                ms[arm].append(round(float(np.median(times)), 3))
        fwd, bwd = critic_launches(pmb.critic, batch)
        key = "%s_B%d_T%d" % (shape_key, B, T)
        record["configs"][key] = {"step_ms": ms, "critic_launches_one_step": {"forward": fwd, "backward": bwd}}
        print(key, json.dumps(record["configs"][key]), flush=True)
    if a.out:
        with open(a.out, "w") as f:
            json.dump(record, f, indent=1)
    print(json.dumps(record))


if __name__ == "__main__":
    main()
