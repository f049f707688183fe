"""Custom-learner step through the modules' autograd path (args.autograd_modules) against the same learner on plain torch.

The step is the one tests/test_module_autograd.py checks against the fused learner step: learners/q_learner.py:37-103
restated on a MAC, a target MAC, a mixer and a target mixer, forward + loss.backward(), no optimiser.  Two arms on the same
GPU and the same data:
  pmb    BasicMAC / QMixer / VDNMixer of this package with autograd_modules = True (one autograd node per timestep,
         pmb_agent_step_bwd / pmb_mixer_bwd in the backward)
  torch  nn.Linear / nn.GRUCell / the reference QMixer in fp32 on the GPU, inputs built with torch ops per timestep
Each step is timed with CUDA events; the arms alternate within every round.  The library launches per timestep of the MAC
forward and backward are counted with pmb_launch_count.  The card name, power limit and SM clock are read in the same run.

    python tools/autograd_bench.py --steps 20 --warmup 3 --out profiles/r05_autograd.json
"""
import argparse
import copy
import json
import os
import subprocess
import sys

import numpy as np
import torch as th

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.join(REPO, "tests"))

from test_module_autograd import RefAgent, RefQMixer, custom_q_learner_backward  # noqa: E402
from cuda_utils import to_batch  # noqa: E402
from pymarl_b200 import _lib, mac_REGISTRY  # noqa: E402
from pymarl_b200.modules.mixers.qmix import QMixer  # noqa: E402
from pymarl_b200.synthetic import SMAC_SHAPES, default_args, make_scheme, torch_episode_fields  # noqa: E402

CONFIGS = [("3m", 32, 60), ("2s3z", 128, 120)]


class TorchMAC:
    """BasicMAC.forward on plain torch modules (basic_controller.py:40-49,100-135)."""

    def __init__(self, agent, args):
        self.agent, self.args = agent, args

    def init_hidden(self, bs):
        self.h = th.zeros(bs * self.args.n_agents, self.args.rnn_hidden_dim, device="cuda")

    def forward(self, batch, t):
        obs = batch["obs"][:, t]
        B, N, A = obs.shape[0], obs.shape[1], self.args.n_actions
        oh = th.zeros(B, N, A, device="cuda")
        if t > 0:
            oh.scatter_(2, batch["actions"][:, t - 1], 1.0)
            oh *= batch["filled"][:, t - 1, None].float()
        x = th.cat([obs, oh, th.eye(N, device="cuda").expand(B, N, N)], -1).reshape(B * N, -1)
        q, self.h = self.agent(x, self.h)
        return q.view(B, N, A)


def _gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader,nounits", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip().split(", ")
        return dict(zip(q.split(","), out))
    except Exception as ex:                      # reported, not fatal
        return {"error": repr(ex)[:200]}


def build_arms(shape_key):
    shape = SMAC_SHAPES[shape_key]
    args = default_args(shape, mixer="qmix", device="cuda", autograd_modules=True)
    scheme, groups = make_scheme(shape)
    mac = mac_REGISTRY["basic_mac"](scheme, groups, args)
    mac.cuda()
    target_mac = copy.deepcopy(mac)
    mixer, target_mixer = QMixer(args).cuda(), QMixer(args).cuda()
    target_mixer.load_state_dict(mixer.state_dict())
    pmb = (mac, target_mac, mixer, target_mixer)
    t_agent = RefAgent(mac.agent.d_in, args.rnn_hidden_dim, args.n_actions).cuda()
    t_agent.load_state_dict(mac.agent.state_dict())
    t_mixer = RefQMixer(shape.state_dim, shape.n_agents, args.mixing_embed_dim).cuda()
    t_mixer.load_state_dict(mixer.state_dict())
    t_target_mixer = copy.deepcopy(t_mixer)
    t_agent_tg = copy.deepcopy(t_agent)
    torch_arm = (TorchMAC(t_agent, args), TorchMAC(t_agent_tg, args), t_mixer, t_target_mixer)
    params = {"pmb": list(mac.agent.parameters()) + list(mixer.parameters()),
              "torch": list(t_agent.parameters()) + list(t_mixer.parameters())}
    return args, {"pmb": pmb, "torch": torch_arm}, params


class Batch:
    def __init__(self, fields, B, T):
        self.fields, self.batch_size, self.max_seq_length = fields, B, T

    def __getitem__(self, k):
        return self.fields[k]


def mac_launches(mac, batch, T):
    """Library launches per timestep of the MAC forward and of its backward."""
    L = _lib.lib()
    th.cuda.synchronize()
    n0 = L.pmb_launch_count()
    mac.init_hidden(batch.batch_size)
    loss = sum(mac.forward(batch, t).sum() for t in range(T))
    n1 = L.pmb_launch_count()
    loss.backward()
    n2 = L.pmb_launch_count()
    for p in mac.agent.parameters():
        p.grad = None
    return (n1 - n0) / T, (n2 - n1) / T


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    assert th.cuda.is_available(), "autograd_bench needs a CUDA device"
    record = {"what": "custom learner step (q_learner.py:37-103 on the modules, forward + loss.backward(), no optimiser), "
                      "QMIX, double_q, ragged episodes; median ms per step over --steps CUDA-event-timed steps per round",
              "steps": a.steps, "warmup": a.warmup, "rounds": a.rounds, "gpu": _gpu_info(), "configs": {}}
    for shape_key, B, T in CONFIGS:
        args, arms, params = build_arms(shape_key)
        fields = torch_episode_fields(SMAC_SHAPES[shape_key], B, T, seed=1, ragged=True, with_onehot=False)
        batch = to_batch(SMAC_SHAPES[shape_key], {k: v.cpu().numpy() for k, v in fields.items()})
        ms = {"pmb": [], "torch": []}

        def step(arm):
            for p in params[arm]:
                p.grad = None
            custom_q_learner_backward(*arms[arm], batch if arm == "pmb" else Batch(fields, B, T), args)

        for arm in ms:
            for _ in range(a.warmup):
                step(arm)
        th.cuda.synchronize()
        for _ in range(a.rounds):
            for arm in ms:
                times = []
                for _ in range(a.steps):
                    e0, e1 = th.cuda.Event(enable_timing=True), th.cuda.Event(enable_timing=True)
                    e0.record()
                    step(arm)
                    e1.record()
                    e1.synchronize()
                    times.append(e0.elapsed_time(e1))
                ms[arm].append(round(float(np.median(times)), 3))
        fwd, bwd = mac_launches(arms["pmb"][0], batch, T)
        record["configs"]["%s_B%d_T%d" % (shape_key, B, T)] = {
            "step_ms": ms, "mac_launches_per_timestep": {"forward": fwd, "backward": bwd}}
        print(shape_key, B, T, json.dumps(record["configs"]["%s_B%d_T%d" % (shape_key, B, T)]), flush=True)
    if a.out:
        with open(a.out, "w") as f:
            json.dump(record, f, indent=1)
    print(json.dumps(record))


if __name__ == "__main__":
    main()
