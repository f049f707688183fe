"""Reference-typed against compact state / avail_actions storage (pmb_batch.state_dtype / avail_dtype).

Both arms store obs as bf16.  Arm "ref" stores state as fp32 and avail_actions as int32 (the reference's types); arm
"compact" stores state as bf16 and avail_actions as uint8.  Both hold the same values (state rounded to bf16), so their
outputs must be bit-identical; every workload checks that.  The arms alternate --rounds times in every measurement.

Workloads (27m_vs_30m, QMIX, bf16 tier):
  1. host zero-copy sample + train: B = --host-batch episodes of a pinned host ReplayBuffer of --buffer episodes, T = 180,
     zero_copy, 512-episode chunks gathered over PCIe by the kernel; full-length episodes, and ragged ones with
     args.skip_padded_steps (the arms of tools/host_replay_bench.py).  Host clock around sample + train, ending in a
     device synchronise.
  2. the learner step on a device batch of --batch episodes (CUDA events around --steps steps).
  3. select_actions for --envs envs x 27 agents (CUDA events around 50 steps, in-kernel draws).
Rates are GB/s over the bytes computed from the shapes: the fields each workload reads (workload 1: the bytes the
sample moves over PCIe, each episode's first F_j = min(T, l_j + 2) steps when trimming; workload 2: every field the step
reads, B x T steps; workload 3: obs and avail of the step, actions and filled of the step before, and the fp32 hidden state in and out).
The card name, power limit and SM clock are read in the same run.

    python tools/compact_fields_bench.py [--rounds 3] [--out FILE]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

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
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--T", type=int, default=180)
    ap.add_argument("--host-batch", type=int, default=1024)
    ap.add_argument("--buffer", type=int, default=1280)
    ap.add_argument("--host-iters", type=int, default=2)
    ap.add_argument("--batch", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--envs", type=int, default=16384)
    ap.add_argument("--workloads", default="host,device,rollout")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()

    import numpy as np
    import torch as th
    if not th.cuda.is_available():
        raise SystemExit("compact_fields_bench: no CUDA device (timings are only meaningful on the GPU)")
    from cuda_utils import Logger
    from pymarl_b200 import le_REGISTRY, mac_REGISTRY
    from pymarl_b200.components.episode_buffer import ReplayBuffer
    from pymarl_b200.components.transforms import OneHot
    from pymarl_b200.synthetic import SMAC_SHAPES, default_args, make_scheme, torch_episode_fields

    shape = SMAC_SHAPES["27m_vs_30m"]
    N, O, S, A, T = shape.n_agents, shape.obs_dim, shape.state_dim, shape.n_actions, a.T
    DT = {"ref": {"state": th.float32, "avail_actions": th.int32},
          "compact": {"state": th.bfloat16, "avail_actions": th.uint8}}
    arms = list(DT)

    def step_bytes(arm):         # bytes per episode-step of the fields the learner reads
        es = {th.float32: 4, th.int32: 4, th.bfloat16: 2, th.uint8: 1}
        return {"obs": N * O * 2, "state": S * es[DT[arm]["state"]], "avail_actions": N * A * es[DT[arm]["avail_actions"]],
                "actions": N * 8, "reward": 4, "terminated": 1, "filled": 8}

    def rounded(f):
        f["obs"] = f["obs"].to(th.bfloat16)
        f["state"] = f["state"].to(th.bfloat16).float()
        return f

    args = default_args(shape, mixer="qmix", device="cuda", use_cuda=True, learner_log_interval=10 ** 12, precision="bf16",
                        host_stream_chunk=512)
    th.manual_seed(7)
    sch, grp = make_scheme(shape)
    sch["actions_onehot"] = {"vshape": (A,), "dtype": th.float32, "group": "agents"}
    learner = le_REGISTRY["q_learner"](mac_REGISTRY["basic_mac"](sch, grp, args), sch, Logger(), args)
    learner.cuda()
    p0 = {k: learner._ensure_flat()[k].clone() for k in ("p", "sq", "target")}

    def restore():
        for k, v in p0.items():
            learner._flat[k].copy_(v)

    def outputs(fn):
        restore()
        fn()
        th.cuda.synchronize()
        return learner._flat["p"].clone(), learner.last_stats.clone()

    def timed(fn, n):
        e0, e1 = th.cuda.Event(enable_timing=True), th.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(n):
            fn(i)
        e1.record()
        th.cuda.synchronize()
        return e0.elapsed_time(e1) / n

    def wall(fn, n):
        th.cuda.synchronize()
        t = time.perf_counter()
        for i in range(n):
            fn(i)
        th.cuda.synchronize()
        return (time.perf_counter() - t) * 1e3 / n

    def alternate(make, steps, warmup, clock, nbytes):
        ms = {k: [] for k in arms}
        for _ in range(a.rounds):
            for arm in arms:
                fn = make(arm)
                clock(fn, warmup)
                ms[arm].append(clock(fn, steps))
        r = {"ms_" + k: [round(x, 3) for x in v] for k, v in ms.items()}
        for k, v in ms.items():
            r["median_ms_" + k] = round(statistics.median(v), 3)
            r["bytes_" + k] = nbytes[k]
            r["GBps_" + k] = round(nbytes[k] / statistics.median(v) / 1e6, 2)
        r["ratio_compact_ref"] = round(r["median_ms_compact"] / r["median_ms_ref"], 4)
        r["byte_ratio_compact_ref"] = round(nbytes["compact"] / nbytes["ref"], 4)
        return r

    rec = {"config": "27m_vs_30m qmix bf16 tier, bf16 obs in both arms", "T": T, "rounds": a.rounds, "gpu": _gpu_info(),
           "dtypes": {k: {f: str(t).replace("torch.", "") for f, t in v.items()} for k, v in DT.items()},
           "step_bytes": {k: sum(step_bytes(k).values()) for k in arms}}
    todo = a.workloads.split(",")

    # 1. host zero-copy sample + train
    if "host" in todo:
        Bh, nb = a.host_batch, a.buffer
        rec["host_zero_copy"] = {"B": Bh, "buffer_episodes": nb, "chunk": 512}
        for ragged in (False, True):
            learner.args.skip_padded_steps = ragged
            bufs = {}
            for arm in arms:
                scheme, groups = make_scheme(shape)
                scheme["obs"]["dtype"] = th.bfloat16
                for k, v in DT[arm].items():
                    scheme[k]["dtype"] = v
                bufs[arm] = ReplayBuffer(scheme, groups, nb, T, {"actions": ("actions_onehot", [OneHot(out_dim=A)])}, "cpu",
                                         pin_memory=True)
            for c0 in range(0, nb, 256):
                c1 = min(nb, c0 + 256)
                f = rounded(torch_episode_fields(shape, c1 - c0, T, seed=1000 + c0, ragged=ragged, device="cuda"))
                for buf in bufs.values():
                    for k, v in f.items():
                        buf.data.transition_data[k][c0:c1].copy_(v)
                del f
            for buf in bufs.values():
                buf.episodes_in_buffer, buf.buffer_index, buf.zero_copy = nb, 0, True
            th.cuda.synchronize()
            np.random.seed(0)
            ids = np.random.choice(nb, Bh, replace=False)
            fl = bufs["ref"].data.transition_data["filled"][th.as_tensor(ids), :, 0].numpy()
            last = np.where(fl.any(1), T - 1 - np.argmax(fl[:, ::-1] != 0, axis=1), -1)
            F = np.where(last < 0, 0, np.minimum(T, last + 2)) if ragged else np.full(Bh, T)
            nbytes = {k: int(F.sum()) * sum(step_bytes(k).values()) for k in arms}

            def make(arm):
                def fn(i):
                    np.random.seed(0)              # the same sample every iteration: the byte count above holds
                    s = bufs[arm].sample(Bh)
                    learner.train(s[:, :s.max_t_filled()], 0, 0)
                return fn

            r = alternate(make, a.host_iters, 1, wall, nbytes)
            r["live_step_fraction"] = round(float(F.sum()) / (Bh * T), 4)
            outs = [outputs(lambda: make(arm)(0)) for arm in arms]
            r["outputs_bit_identical"] = bool(th.equal(outs[0][0], outs[1][0]) and th.equal(outs[0][1], outs[1][1]))
            rec["host_zero_copy"]["ragged_skip" if ragged else "full"] = r
            print(json.dumps({"host_zero_copy": {"ragged" if ragged else "full": r}}), flush=True)
            del bufs
        learner.args.skip_padded_steps = False
        restore()

    # 2. device-batch learner step
    if "device" in todo:
        B = a.batch
        f = rounded(torch_episode_fields(shape, B, T, seed=4242, ragged=False, device="cuda", with_onehot=False))
        dev = {"ref": _DictBatch(f, B, T),
               "compact": _DictBatch(dict(f, state=f["state"].to(th.bfloat16), avail_actions=f["avail_actions"].to(th.uint8)),
                                     B, T)}
        nbytes = {k: B * T * sum(step_bytes(k).values()) for k in arms}
        r = alternate(lambda arm: (lambda i: learner.train(dev[arm], i, 0)), a.steps, a.warmup, timed, nbytes)
        r["B"] = B
        outs = [outputs(lambda: learner.train(dev[arm], 0, 0)) for arm in arms]
        r["outputs_bit_identical"] = bool(th.equal(outs[0][0], outs[1][0]) and th.equal(outs[0][1], outs[1][1]))
        rec["device_batch_train"] = r
        print(json.dumps({"device_batch_train": r}), flush=True)
        restore()
        del dev, f
        th.cuda.empty_cache()

    # 3. rollout
    if "rollout" in todo:
        E = a.envs
        rf = torch_episode_fields(shape, E, 4, seed=99, ragged=False, device="cuda", with_onehot=False)
        rf["obs"] = rf["obs"].to(th.bfloat16)
        rb = {"ref": _DictBatch(rf, E, 4), "compact": _DictBatch(dict(rf, avail_actions=rf["avail_actions"].to(th.uint8)), E, 4)}
        mac = learner.mac

        def step(arm):
            def fn(i):
                if i == 0:
                    mac.init_hidden(E)
                mac._run_step(rb[arm], 1, epsilon=0.05, seed=1, offset=i, want_actions=True, want_q=False)
            return fn

        R = E * N
        nbytes = {k: R * (O * 2 + A * (4 if k == "ref" else 1) + 8) + E * 8 + 2 * R * 64 * 4 for k in arms}
        r = alternate(step, 50, 5, timed, nbytes)
        r["envs"], r["agents"] = E, N
        acts = {}
        for arm in arms:
            mac.init_hidden(E)
            _, acts[arm] = mac._run_step(rb[arm], 1, epsilon=0.05, seed=1, offset=0, want_actions=True, want_q=False)
        r["actions_bit_identical"] = bool(th.equal(acts["ref"], acts["compact"]))
        rec["select_actions"] = r
        print(json.dumps({"select_actions": r}), flush=True)

    rec["gpu_after"] = _gpu_info()
    line = json.dumps(rec)
    print(line)
    if a.out:
        with open(a.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
