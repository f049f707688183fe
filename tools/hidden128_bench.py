"""The learner step and the rollout step at rnn_hidden_dim 64 and 128, on both precision tiers.

Workload: QMIX, 27m_vs_30m, B = 1024 full-length episodes of T = 180 (the fp32 activations of the H = 128 learner step are
about 20 GB here, 80 GB at B = 4096), and select_actions for 1024 envs x 27 agents with in-kernel draws.  The four
configurations (tier x H) alternate --rounds times, each with its own warm-up:
- learner step: ms / step from CUDA events around --steps steps on the same device batch;
- rollout step: ms / step from CUDA events around --rollout-steps steps;
- the per-phase times of one profiled learner step and one profiled rollout step per configuration and round
  (pmb_profile_begin / end), in launch order (at H = 128 the gi GEMM / recurrence / fc2 GEMM phases come once for the
  target net, then once for the online net).  The rollout step's last phase (fc2 and the selection) is not closed by
  a mark: its time is the step time less the phases listed.
The card name, power limit and SM clock are read in the same run.

    python tools/hidden128_bench.py [--steps 10] [--warmup 2] [--rounds 3] [--out FILE]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.join(REPO, "tests"))


class _DictBatch:
    def __init__(self, fields, batch_size, max_seq_length):
        self.fields, self.batch_size, self.max_seq_length = fields, batch_size, max_seq_length
        self.device = next(iter(fields.values())).device

    def __getitem__(self, k):
        return self.fields[k]


def _gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader,nounits", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip().split(", ")
        return dict(zip(q.split(","), out))
    except Exception as ex:                      # reported, not fatal
        return {"error": repr(ex)[:200]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--rollout-steps", type=int, default=50)
    ap.add_argument("--batch", type=int, default=1024)
    ap.add_argument("--T", type=int, default=180)
    ap.add_argument("--envs", type=int, default=1024)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()

    import torch as th
    if not th.cuda.is_available():
        raise SystemExit("hidden128_bench: no CUDA device (timings are only meaningful on the GPU)")
    from cuda_utils import Logger
    from pymarl_b200 import _lib, le_REGISTRY, mac_REGISTRY
    from pymarl_b200.synthetic import SMAC_SHAPES, default_args, make_scheme, torch_episode_fields

    shape = SMAC_SHAPES["27m_vs_30m"]
    B, T, E = a.batch, a.T, a.envs
    fields = torch_episode_fields(shape, B, T, seed=4242, ragged=False, device="cuda", with_onehot=False)
    batch = _DictBatch(fields, B, T)
    rf = torch_episode_fields(shape, E, 4, seed=99, ragged=False, device="cuda", with_onehot=False)
    rbatch = _DictBatch(rf, E, 4)

    configs = {}
    for precision in ("fp32", "bf16"):
        for H in (64, 128):
            args = default_args(shape, mixer="qmix", device="cuda", use_cuda=True, learner_log_interval=10 ** 12,
                                precision=precision, rnn_hidden_dim=H)
            th.manual_seed(7)
            scheme, groups = make_scheme(shape)
            scheme["actions_onehot"] = {"vshape": (shape.n_actions,), "dtype": th.float32, "group": "agents"}
            learner = le_REGISTRY["q_learner"](mac_REGISTRY["basic_mac"](scheme, groups, args), scheme, Logger(), args)
            learner.cuda()
            configs["%s_h%d" % (precision, H)] = learner

    def timed(fn, n):
        e0, e1 = th.cuda.Event(enable_timing=True), th.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(n):
            fn(i)
        e1.record()
        th.cuda.synchronize()
        return e0.elapsed_time(e1) / n

    def rollout(learner):
        mac = learner.mac

        def fn(i):
            if i == 0:
                mac.init_hidden(E)
            mac._run_step(rbatch, 1, epsilon=0.05, seed=1, offset=i, want_actions=True, want_q=False)
        return fn

    def profiled(fn):
        th.cuda.synchronize()
        _lib.profile_begin()
        fn(0)
        return [(name, round(ms, 4)) for name, ms in _lib.profile_end(max_phases=64)]

    rec = {"config": "27m_vs_30m qmix, full-length episodes", "B": B, "T": T, "envs": E, "steps": a.steps,
           "warmup": a.warmup, "rounds": a.rounds, "gpu": _gpu_info(), "learner_ms": {}, "rollout_ms": {},
           "learner_phases_ms": {}, "rollout_phases_ms": {}}
    for k in configs:
        rec["learner_ms"][k], rec["rollout_ms"][k] = [], []
        rec["learner_phases_ms"][k], rec["rollout_phases_ms"][k] = [], []
    for _ in range(a.rounds):
        for k, learner in configs.items():
            train = lambda i, lr=learner: lr.train(batch, i, 0)
            timed(train, a.warmup)
            rec["learner_ms"][k].append(round(timed(train, a.steps), 3))
            rec["learner_phases_ms"][k].append(profiled(train))
            ro = rollout(learner)
            timed(ro, 5)
            rec["rollout_ms"][k].append(round(timed(ro, a.rollout_steps), 4))
            rec["rollout_phases_ms"][k].append(profiled(ro))
    rec["median_learner_ms"] = {k: statistics.median(v) for k, v in rec["learner_ms"].items()}
    rec["median_rollout_ms"] = {k: statistics.median(v) for k, v in rec["rollout_ms"].items()}
    # phases of the last round, summed by name
    rec["learner_phase_sums_ms"] = {}
    for k, runs in rec["learner_phases_ms"].items():
        tot = {}
        for name, ms in runs[-1]:
            tot[name] = round(tot.get(name, 0.0) + ms, 4)
        rec["learner_phase_sums_ms"][k] = tot
    rec["gpu_after"] = _gpu_info()
    s = json.dumps(rec, indent=1)
    print(json.dumps({"median_learner_ms": rec["median_learner_ms"], "median_rollout_ms": rec["median_rollout_ms"],
                      "gpu": rec["gpu"], "learner_phase_sums_ms": rec["learner_phase_sums_ms"]}, indent=1))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
