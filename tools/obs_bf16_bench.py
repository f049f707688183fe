"""fp32-stored against bf16-stored observations (pmb_batch.obs_dtype) at BASELINE config 4.

Workload: QMIX, 27m_vs_30m, B = 4096, T = 180, bf16 tier, full-length episodes from the bench's generator with obs rounded
to bf16, so that both arms hold the same values.  The arms alternate --rounds times (each with its own warm-up) in every
measurement:
- the learner step on a device batch (median ms / step, CUDA events around --steps steps) and the median per-phase times
  of --profiled profiled steps per arm and round (pmb_profile_begin / end; the streaming fc1 is "fc1_fwd_both_tc");
- a zero-copy replay sample (B random episode ids of the device batch as the buffer) + train;
- the host-streamed step (host-resident batch of --host-batch episodes, 512-episode chunks);
- select_actions for 16384 envs x 27 agents (in-kernel draws).
Outputs are checked: the updated parameters and loss sums of one step from the same start, and the rollout's actions,
must be bit-identical between the arms.  The card name, power limit and SM clock are read in the same run.

    python tools/obs_bf16_bench.py [--steps 20] [--warmup 3] [--rounds 3] [--out FILE]
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


class _Sample:
    """What ReplayBuffer.sample returns for zero-copy sampling: episode ids into a buffer that stays where it is."""
    def __init__(self, fields, ep_ids, max_seq_length):
        from types import SimpleNamespace
        self.buffer = SimpleNamespace(data=SimpleNamespace(transition_data=fields))
        self.ep_ids, self.batch_size, self.max_seq_length = ep_ids, int(ep_ids.numel()), max_seq_length


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
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--profiled", type=int, default=3)
    ap.add_argument("--batch", type=int, default=4096)
    ap.add_argument("--T", type=int, default=180)
    ap.add_argument("--host-batch", type=int, default=1024)
    ap.add_argument("--host-steps", type=int, default=2)
    ap.add_argument("--envs", type=int, default=16384)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()

    import torch as th
    if not th.cuda.is_available():
        raise SystemExit("obs_bf16_bench: no CUDA device (timings are only meaningful on the GPU)")
    from cuda_utils import Logger
    from pymarl_b200 import _lib, le_REGISTRY, mac_REGISTRY
    from pymarl_b200.synthetic import SMAC_SHAPES, default_args, make_scheme, torch_episode_fields

    shape = SMAC_SHAPES["27m_vs_30m"]
    B, T = a.batch, a.T
    args = default_args(shape, mixer="qmix", device="cuda", use_cuda=True, learner_log_interval=10 ** 12, precision="bf16")
    th.manual_seed(7)
    scheme, groups = make_scheme(shape)
    scheme["actions_onehot"] = {"vshape": (shape.n_actions,), "dtype": th.float32, "group": "agents"}
    learner = le_REGISTRY["q_learner"](mac_REGISTRY["basic_mac"](scheme, groups, args), scheme, Logger(), args)
    learner.cuda()
    p0 = {k: learner._ensure_flat()[k].clone() for k in ("p", "sq", "target")}

    def restore():
        for k, v in p0.items():
            learner._flat[k].copy_(v)

    f32 = torch_episode_fields(shape, B, T, seed=4242, ragged=False, device="cuda", with_onehot=False)
    f32["obs"] = f32["obs"].to(th.bfloat16).float()
    f16 = dict(f32)
    f16["obs"] = f32["obs"].to(th.bfloat16)
    arms = {"fp32": f32, "bf16": f16}
    ids = th.randperm(B, device="cuda")

    def timed(fn, n):
        e0, e1 = th.cuda.Event(enable_timing=True), th.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(n):
            fn(i)
        e1.record()
        th.cuda.synchronize()
        return e0.elapsed_time(e1) / n

    def alternate(make, steps, warmup):
        ms = {k: [] for k in arms}
        for _ in range(a.rounds):
            for arm in arms:
                fn = make(arm)
                timed(fn, warmup)
                ms[arm].append(timed(fn, steps))
        return {"ms_" + k: [round(x, 3) for x in v] for k, v in ms.items()} | \
               {"median_ms_" + k: round(statistics.median(v), 3) for k, v in ms.items()}

    def profiled(batch):
        th.cuda.synchronize()
        _lib.profile_begin()
        learner.train(batch, 0, 0)
        out = {}
        for name, ms in _lib.profile_end(max_phases=64):
            out[name] = round(out.get(name, 0.0) + ms, 4)
        return out

    def outputs(batch):
        restore()
        learner.train(batch, 0, 0)
        th.cuda.synchronize()
        return learner._flat["p"].clone(), learner.last_stats.clone()

    rec = {"config": "27m_vs_30m qmix bf16 tier, full-length episodes", "B": B, "T": T, "steps": a.steps, "warmup": a.warmup,
           "rounds": a.rounds, "gpu": _gpu_info(),
           "obs_bytes": {k: v["obs"].numel() * v["obs"].element_size() for k, v in arms.items()}}

    # 1. device batch
    dev = {k: _DictBatch(v, B, T) for k, v in arms.items()}
    rec["train"] = alternate(lambda arm: (lambda i: learner.train(dev[arm], i, 0)), a.steps, a.warmup)
    # per-phase times: --profiled steps per arm and round, arms alternated; medians over all of them
    runs = {k: [] for k in arms}
    for _ in range(a.rounds):
        for k in arms:
            runs[k] += [profiled(dev[k]) for _ in range(a.profiled)]
    ph = {k: {n: round(statistics.median(r[n] for r in runs[k]), 4) for n in runs[k][0]} for k in arms}
    rec["train"]["phases_ms_median"] = ph
    rec["train"]["fc1_ms_all"] = {k: [r.get("fc1_fwd_both_tc") for r in runs[k]] for k in arms}
    rec["train"]["fc1_ms"] = {k: ph[k].get("fc1_fwd_both_tc") for k in arms}
    (p_a, s_a), (p_b, s_b) = outputs(dev["fp32"]), outputs(dev["bf16"])
    rec["train"]["outputs_bit_identical"] = bool(th.equal(p_a, p_b) and th.equal(s_a, s_b))

    # 2. zero-copy sample from the device batch as the buffer
    smp = {k: _Sample(v, ids, T) for k, v in arms.items()}
    rec["zero_copy_sample_train"] = alternate(lambda arm: (lambda i: learner.train(smp[arm], i, 0)), a.steps, a.warmup)
    (p_a, s_a), (p_b, s_b) = outputs(smp["fp32"]), outputs(smp["bf16"])
    rec["zero_copy_sample_train"]["outputs_bit_identical"] = bool(th.equal(p_a, p_b) and th.equal(s_a, s_b))
    restore()
    del dev, smp
    th.cuda.empty_cache()

    # 3. host-streamed step
    Bh = a.host_batch
    host = {k: _DictBatch({n: t[:Bh].cpu() for n, t in v.items()}, Bh, T) for k, v in arms.items()}
    args.host_stream_chunk = 512
    rec["host_streamed"] = {"B": Bh, "chunk": 512}
    rec["host_streamed"] |= alternate(lambda arm: (lambda i: learner.train(host[arm], i, 0)), a.host_steps, 1)
    (p_a, s_a), (p_b, s_b) = outputs(host["fp32"]), outputs(host["bf16"])
    rec["host_streamed"]["outputs_bit_identical"] = bool(th.equal(p_a, p_b) and th.equal(s_a, s_b))
    restore()
    del host
    del f32, f16, arms
    th.cuda.empty_cache()

    # 4. rollout: select_actions for --envs envs
    E, Tr = a.envs, 4
    rf = torch_episode_fields(shape, E, Tr, seed=99, ragged=False, device="cuda", with_onehot=False)
    ro32 = rf["obs"].to(th.bfloat16).float()
    arms = {"fp32": ro32, "bf16": ro32.to(th.bfloat16)}
    mac = learner.mac

    class _RB:
        def __init__(self, obs):
            self.f = dict(rf, obs=obs)
            self.batch_size, self.device = E, obs.device

        def __getitem__(self, k):
            return self.f[k]

    rb = {k: _RB(v) for k, v in arms.items()}

    def step(arm):
        def fn(i):
            if i == 0:
                mac.init_hidden(E)
            mac._run_step(rb[arm], 1, epsilon=0.05, seed=1, offset=i, want_actions=True, want_q=False)
        return fn

    rec["select_actions"] = {"envs": E, "agents": shape.n_agents}
    rec["select_actions"] |= alternate(step, 50, 5)
    acts = {}
    for arm in rb:
        mac.init_hidden(E)
        _, acts[arm] = mac._run_step(rb[arm], 1, epsilon=0.05, seed=1, offset=0, want_actions=True, want_q=False)
    rec["select_actions"]["actions_bit_identical"] = bool(th.equal(acts["fp32"], acts["bf16"]))
    for k in ("train", "zero_copy_sample_train", "host_streamed", "select_actions"):
        r = rec[k]
        r["ratio_bf16_fp32"] = round(r["median_ms_bf16"] / r["median_ms_fp32"], 4)
    rec["gpu_after"] = _gpu_info()
    line = json.dumps(rec)
    print(line)
    if a.out:
        with open(a.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
