"""Sampling + training from a replay buffer in host memory (buffer_cpu_only), today's path against zero-copy sampling.

Workload: QMIX, 27m_vs_30m, bf16 tier, B = 4096 sampled from a buffer of more than B episodes (T = 180), sized to the
host's available memory.  Four data sets: fp32 or bf16 obs, full-length or ragged episodes (ragged: the learner runs with
args.skip_padded_steps, so the gather kernel trims each episode's padded tail).  Per data set the arms alternate
--rounds times:
  (a) today:   unpinned buffer, sample() (host gather of every field), [:, :max_t], train (streamed 512-episode chunks)
  (b) new:     pinned buffer with zero_copy, sample() (ids), [:, :max_t], train (chunks gathered over PCIe by the kernel)
  (c) ceiling: one cudaMemcpyAsync of a contiguous pinned block of the bytes that (b) moves over PCIe
Reported: ms per iteration (host clock around work that ends in a device synchronise), the bytes (b) reads over PCIe,
the gather kernel alone over the same sample (CUDA events, the whole sample into the two chunk buffers, no compute) in
GB/s, and rates as fractions of (c).  Outputs are checked: one step of (a) and (b) from the same start and ids must give
bit-identical parameters and loss sums.  The card name, power limit and SM clock are read in the same run.

    python tools/host_replay_bench.py [--batch 4096] [--rounds 2] [--iters 3] [--out FILE]
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
    ap.add_argument("--batch", type=int, default=4096)
    ap.add_argument("--T", type=int, default=180)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--iters", type=int, default=3, help="timed iterations of arms (b) and (c) per round")
    ap.add_argument("--iters-a", type=int, default=1, help="timed iterations of arm (a) per round")
    ap.add_argument("--sets", default="fp32_full,bf16_full,fp32_ragged,bf16_ragged")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()

    import numpy as np
    import psutil
    import torch as th
    if not th.cuda.is_available():
        raise SystemExit("host_replay_bench: no CUDA device (timings are only meaningful on the GPU)")
    from cuda_utils import Logger
    from pymarl_b200 import _lib, le_REGISTRY, mac_REGISTRY
    from pymarl_b200.components.episode_buffer import ReplayBuffer
    from pymarl_b200.components.transforms import OneHot
    from pymarl_b200.synthetic import SMAC_SHAPES, default_args, make_scheme, torch_episode_fields

    shape = SMAC_SHAPES["27m_vs_30m"]
    B, T = a.batch, a.T
    N, O, S, A = shape.n_agents, shape.obs_dim, shape.state_dim, shape.n_actions
    read = ["obs", "actions", "avail_actions", "reward", "terminated", "filled", "state"]
    rec = {"config": "27m_vs_30m qmix bf16 tier, host replay buffer", "B": B, "T": T, "rounds": a.rounds,
           "iters_b_c": a.iters, "iters_a": a.iters_a, "chunk": 512, "gpu": _gpu_info(), "sets": {}}

    th.manual_seed(7)
    for name in a.sets.split(","):
        obs_dtype = th.bfloat16 if name.startswith("bf16") else th.float32
        ragged = name.endswith("ragged")
        scheme, groups = make_scheme(shape)
        scheme["obs"]["dtype"] = obs_dtype
        pre = {"actions": ("actions_onehot", [OneHot(out_dim=A)])}
        step_bytes = {"obs": N * O * (2 if obs_dtype == th.bfloat16 else 4), "actions": N * 8, "avail_actions": N * A * 4,
                      "reward": 4, "terminated": 1, "filled": 8, "state": S * 4}
        ep_bytes = T * (sum(step_bytes.values()) + N * A * 4)                  # + actions_onehot, stored, not read
        avail = psutil.virtual_memory().available
        # two buffers + the gathered sample of arm (a) + the ceiling block of arm (c), with 15 % headroom
        n_buf = min(B + B // 4, int((0.85 * avail - 2 * B * ep_bytes) // (2 * ep_bytes)))
        if n_buf <= B:
            raise MemoryError("host has %.0f GB available; %s needs more than %.0f GB" %
                              (avail / 1e9, name, (2 * (B + 1) + 2 * B) * ep_bytes / 1e9))
        args = default_args(shape, mixer="qmix", device="cuda", use_cuda=True, learner_log_interval=10 ** 12,
                            precision="bf16", host_stream_chunk=512, skip_padded_steps=ragged)
        sch, grp = make_scheme(shape)
        sch["actions_onehot"] = {"vshape": (A,), "dtype": th.float32, "group": "agents"}
        learner = le_REGISTRY["q_learner"](mac_REGISTRY["basic_mac"](sch, grp, args), sch, Logger(), args)
        learner.cuda()
        p0 = {k: learner._ensure_flat()[k].clone() for k in ("p", "sq", "target")}

        t0 = time.time()
        plain = ReplayBuffer(scheme, groups, n_buf, T, pre, "cpu")
        pinned = ReplayBuffer(scheme, groups, n_buf, T, pre, "cpu", pin_memory=True)
        for c0 in range(0, n_buf, 256):
            c1 = min(n_buf, c0 + 256)
            f = torch_episode_fields(shape, c1 - c0, T, seed=1000 + c0, ragged=ragged, device="cuda")
            for buf in (plain, pinned):
                for k, v in f.items():
                    buf.data.transition_data[k][c0:c1].copy_(v)
            del f
        for buf in (plain, pinned):
            buf.episodes_in_buffer, buf.buffer_index = n_buf, 0
        pinned.zero_copy = True
        th.cuda.synchronize()
        r = {"buffer_episodes": n_buf, "buffer_gb_each": round(n_buf * ep_bytes / 1e9, 2),
             "host_available_gb": round(avail / 1e9, 1), "fill_s": round(time.time() - t0, 1)}

        # bytes arm (b) reads over PCIe for the sample of seed 0 (each episode's first F_j steps when trimming)
        np.random.seed(0)
        ids = np.random.choice(n_buf, B, replace=False)
        fl = plain.data.transition_data["filled"][th.as_tensor(ids), :, 0].numpy()
        if ragged:
            last = np.where(fl.any(1), T - 1 - np.argmax(fl[:, ::-1] != 0, axis=1), -1)
            F = np.where(last < 0, 0, np.minimum(T, last + 2))
        else:
            F = np.full(B, T)
        pcie = int(F.sum()) * sum(step_bytes.values())
        r["pcie_bytes"] = pcie
        r["live_step_fraction"] = round(float(F.sum()) / (B * T), 4)

        block = _lib.host_empty((pcie,), th.uint8)
        block.fill_(1)
        dst = th.empty(pcie, dtype=th.uint8, device="cuda")

        it = {"a": 0, "b": 0}

        def arm(key, buf):
            def fn():
                np.random.seed(it[key] % 7)
                it[key] += 1
                s = buf.sample(B)
                learner.train(s[:, :s.max_t_filled()], 0, 0)
            return fn

        def ceiling():
            dst.copy_(block, non_blocking=True)

        def wall(fn, n):
            th.cuda.synchronize()
            t = time.perf_counter()
            for _ in range(n):
                fn()
            th.cuda.synchronize()
            return (time.perf_counter() - t) * 1e3 / n

        arms = {"a_today": (arm("a", plain), a.iters_a), "b_zero_copy": (arm("b", pinned), a.iters),
                "c_ceiling": (ceiling, a.iters)}
        ms = {k: [] for k in arms}
        for _ in range(a.rounds):
            for k, (fn, n) in arms.items():
                fn()                                              # warm-up
                ms[k].append(round(wall(fn, n), 2))
        for k in arms:
            r["ms_" + k] = ms[k]
            r["median_ms_" + k] = statistics.median(ms[k])

        # the gather kernel alone: the whole sample, chunk by chunk into two chunk-sized buffers, CUDA events
        src = {k: pinned.data.transition_data[k] for k in read}
        bufs = [{k: _lib.episode_rows(512, (T,) + tuple(v.shape[2:]), v.dtype, "cuda") for k, v in src.items()}
                for _ in range(2)]
        dev_ids = th.as_tensor(ids, device="cuda")
        trim = src["filled"] if ragged else None

        def gather_all():
            for i, s0 in enumerate(range(0, B, 512)):
                s1 = min(B, s0 + 512)
                _lib.gather_episode_steps(src, dev_ids[s0:s1], T, {k: v[:s1 - s0] for k, v in bufs[i & 1].items()},
                                          filled=trim)

        kms = []
        for _ in range(a.rounds):
            gather_all()
            e0, e1 = th.cuda.Event(enable_timing=True), th.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(a.iters):
                gather_all()
            e1.record()
            th.cuda.synchronize()
            kms.append(round(e0.elapsed_time(e1) / a.iters, 2))
        r["gather_kernel_ms"] = kms
        km = statistics.median(kms)
        c_ms = r["median_ms_c_ceiling"]
        r["gather_kernel_GBps"] = round(pcie / km / 1e6, 2)
        r["ceiling_GBps"] = round(pcie / c_ms / 1e6, 2)
        r["gather_kernel_fraction_of_ceiling"] = round(c_ms / km, 4)
        r["b_fraction_of_ceiling"] = round(c_ms / r["median_ms_b_zero_copy"], 4)
        r["speedup_b_over_a"] = round(r["median_ms_a_today"] / r["median_ms_b_zero_copy"], 2)

        # outputs: one step of (a) and (b) from the same start and the same ids
        outs = []
        for buf in (plain, pinned):
            for k, v in p0.items():
                learner._flat[k].copy_(v)
            np.random.seed(0)
            s = buf.sample(B)
            learner.train(s[:, :s.max_t_filled()], 0, 0)
            th.cuda.synchronize()
            outs.append((learner._flat["p"].clone(), learner.last_stats.clone()))
        r["outputs_bit_identical"] = bool(th.equal(outs[0][0], outs[1][0]) and th.equal(outs[0][1], outs[1][1]))
        rec["sets"][name] = r
        print(json.dumps({name: r}), flush=True)
        del plain, pinned, block, dst, bufs, src, learner, outs, trim
        th.cuda.empty_cache()

    rec["gpu_after"] = _gpu_info()
    line = json.dumps(rec)
    print(line)
    if a.out:
        with open(a.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
